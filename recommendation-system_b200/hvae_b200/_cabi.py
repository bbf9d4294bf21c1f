"""ctypes binding of libhvae_b200.so, generated from include/hvae_b200.h at import time.

There is deliberately no fallback: if the shared library is missing or a symbol declared in the header is
not exported, importing this module raises.  Every call returns a status that is turned into RuntimeError
with the library's own message.
"""
from __future__ import annotations

import ctypes
import re
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libhvae_b200.so"
HEADER_PATH = _PKG.parents[1] / "include" / "hvae_b200.h"

_SCALARS = {
    "int": ctypes.c_int, "int32_t": ctypes.c_int32, "int64_t": ctypes.c_int64, "uint32_t": ctypes.c_uint32,
    "uint64_t": ctypes.c_uint64, "float": ctypes.c_float, "double": ctypes.c_double, "size_t": ctypes.c_size_t,
}


def parse_header(path: Path = HEADER_PATH):
    """-> {name: (restype, [argtypes])} for every function declared in the public header."""
    text = re.sub(r"/\*.*?\*/", "", path.read_text(), flags=re.S)
    text = re.sub(r"typedef struct.*?\}\s*\w+;", "", text, flags=re.S)
    decls = {}
    for ret, name, args in re.findall(r"\b(int|size_t|const char\*)\s+(hvae_\w+)\s*\(([^)]*)\)\s*;", text):
        argtypes = []
        for a in [s.strip() for s in args.split(",")]:
            if a in ("void", ""):
                continue
            if "*" in a:
                argtypes.append(ctypes.c_void_p)
            else:
                argtypes.append(_SCALARS[a.replace("const ", "").split()[0]])
        restype = {"int": ctypes.c_int, "size_t": ctypes.c_size_t, "const char*": ctypes.c_char_p}[ret]
        decls[name] = (restype, argtypes)
    return decls


class StepState(ctypes.Structure):
    """Mirror of hvae_step_state (include/hvae_b200.h)."""
    _fields_ = [("adam_step", ctypes.c_int32), ("anneal_step", ctypes.c_int32), ("step_size", ctypes.c_float),
                ("bc2_sqrt", ctypes.c_float), ("beta_kl", ctypes.c_float), ("inv_bg", ctypes.c_float),
                ("kl_coef", ctypes.c_float), ("clip_coef", ctypes.c_float), ("grad_norm", ctypes.c_float),
                ("norm2", ctypes.c_float), ("noise_lo", ctypes.c_uint32), ("noise_hi", ctypes.c_uint32)]


STATE_WORDS = ctypes.sizeof(StepState) // 4
STATE_OFF = {name: getattr(StepState, name).offset // 4 for name, _ in StepState._fields_}


# Kernels of ours launched per C-ABI call (library-internal CUB passes are not counted); default 1.
KERNELS_PER_CALL = {"hvae_ln_act_bwd": 2, "hvae_colsum": 2, "hvae_batch_transpose": 4, "hvae_grad_norm_clip": 2,
                    "hvae_metrics_reduce": 2, "hvae_mask_topk": 2, "hvae_mask_topk_filtered": 2, "hvae_mask_topk_sampled": 2, "hvae_w1_plan": 2, "hvae_w1_grad": 2, "hvae_w1_max_work": 0, "hvae_w1_max_partial_rows": 0,
                    "hvae_tc_n_splits": 0, "hvae_tc_grad_splits": 0, "hvae_gemm_tf32_supported": 0, "hvae_tc_score_lse": 2, "hvae_tc_score_lse_grad": 2, "hvae_tc_onepass_subparts": 0, "hvae_h2d_csr_batch": 0, "hvae_d2h_floats": 0, "hvae_mask_topk_chunks": 0, "hvae_tc_topk_splits": 0, "hvae_last_error": 0, "hvae_abi_version": 0, "hvae_tc_duo_max_clusters": 0,
                    "hvae_ln_bwd_workspace_floats": 0, "hvae_batch_temp_bytes": 0}


class _Lib:
    launches = 0   # running count of hvae kernels launched through this binding (bench.py's gpu_launches)

    def __init__(self):
        if not LIB_PATH.exists():
            raise RuntimeError(f"{LIB_PATH} is missing: build it with `python recommendation-system_b200/build.py` "
                               "(there is no CPU or PyTorch fallback)")
        self._dll = ctypes.CDLL(str(LIB_PATH))
        self.decls = parse_header()
        for name, (restype, argtypes) in self.decls.items():
            fn = getattr(self._dll, name)  # AttributeError if the header and the library disagree
            fn.restype, fn.argtypes = restype, argtypes
            if restype is ctypes.c_int and name not in ("hvae_abi_version", "hvae_tc_duo_max_clusters"):
                setattr(self, name[5:], self._checked(fn, name))
            else:
                setattr(self, name[5:], fn)

    def _checked(self, fn, name):
        nk = KERNELS_PER_CALL.get(name, 1)

        def call(*args):
            rc = fn(*args)
            if rc != 0:
                raise RuntimeError(f"{name}: {self._dll.hvae_last_error().decode()}")
            self.launches += nk
        call.__name__ = name
        return call


_lib = None


def lib() -> _Lib:
    global _lib
    if _lib is None:
        _lib = _Lib()
    return _lib


def p(t):
    """Device pointer of a tensor (or NULL)."""
    return None if t is None else t.data_ptr()
