"""Stage sequencing of the HybridVAE hot path over the C ABI (include/hvae_b200.h).

`Layout` places every parameter in one flat fp32 arena (W1^T first, then the small dense tensors) so the
fused Adam and the grad-norm run over contiguous memory.  `Engine` owns the arena-shaped optimiser state,
a grow-only workspace, and issues the kernels of one training step / validation step / scoring pass on
torch's current stream.  PyTorch is used for allocation, streams and CUDA-graph capture only.
"""
from __future__ import annotations

import contextlib
import ctypes
from dataclasses import dataclass

import os

import numpy as np
import torch

from . import _cabi
from ._cabi import STATE_OFF, STATE_WORDS, p


def r4(n: int) -> int:
    return (n + 3) // 4 * 4


def r8(n: int) -> int:
    return (n + 7) // 8 * 8


@dataclass
class Slot:
    off: int      # offset in floats from the arena start
    rows: int
    cols: int
    ld: int       # row stride in floats
    vec: bool = False

    @property
    def size(self):
        return self.rows * self.ld


class Layout:
    """Arena layout.  Reference tensor names (src/ml/model.py state_dict, SURVEY.md §8 a1) map to slots."""

    def __init__(self, n_items: int, emb_dim: int, latent_dim: int, hidden_dims):
        self.N, self.d, self.L, self.hidden = n_items, emb_dim, latent_dim, list(hidden_dims)
        self.identity_proj = latent_dim == emb_dim
        self.slots: dict[str, Slot] = {}
        off = 0

        def add(name, rows, cols):
            nonlocal off
            s = Slot(off, rows, cols, r4(cols), vec=(rows == 1))
            self.slots[name] = s
            off += s.size
            return s

        h = self.hidden
        add("encoder.0.weight", n_items, h[0]).vec = False  # stored TRANSPOSED: [N, ld(h0)]
        self.n_w1 = off
        add("encoder.0.bias", 1, h[0])
        add("encoder.1.weight", 1, h[0])
        add("encoder.1.bias", 1, h[0])
        for i in range(1, len(h)):
            add(f"encoder.{4 * i}.weight", h[i], h[i - 1]).vec = False
            add(f"encoder.{4 * i}.bias", 1, h[i])
            add(f"encoder.{4 * i + 1}.weight", 1, h[i])
            add(f"encoder.{4 * i + 1}.bias", 1, h[i])
        add("fc_mu.weight", latent_dim, h[-1]).vec = False  # fc_mu / fc_logvar adjacent: one [2L, h] GEMM
        add("fc_logvar.weight", latent_dim, h[-1]).vec = False
        self.slots["fc_ml.bias"] = Slot(off, 1, 2 * latent_dim, r4(2 * latent_dim))
        off += r4(2 * latent_dim)
        if not self.identity_proj:
            add("projection_layer.0.weight", emb_dim, latent_dim).vec = False
            add("projection_layer.0.bias", 1, emb_dim)
            add("projection_layer.3.weight", emb_dim, emb_dim).vec = False
            add("projection_layer.3.bias", 1, emb_dim)
        self.n_params = off
        self.n_dense = off - self.n_w1

    def reference_keys(self):
        keys = ["encoder.0.weight", "encoder.0.bias", "encoder.1.weight", "encoder.1.bias"]
        for i in range(1, len(self.hidden)):
            keys += [f"encoder.{4 * i}.weight", f"encoder.{4 * i}.bias", f"encoder.{4 * i + 1}.weight",
                     f"encoder.{4 * i + 1}.bias"]
        keys += ["fc_mu.weight", "fc_mu.bias", "fc_logvar.weight", "fc_logvar.bias"]
        if not self.identity_proj:
            keys += ["projection_layer.0.weight", "projection_layer.0.bias", "projection_layer.3.weight",
                     "projection_layer.3.bias"]
        return keys

    # -- views in reference shapes ----------------------------------------------------------------------
    def view(self, arena: torch.Tensor, key: str) -> torch.Tensor:
        """Reference-shaped *view* (no copy) of one tensor inside an arena-shaped buffer."""
        L = self.L
        if key in ("fc_mu.bias", "fc_logvar.bias"):
            s = self.slots["fc_ml.bias"]
            o = s.off + (0 if key == "fc_mu.bias" else L)
            return arena[o:o + L]
        s = self.slots[key]
        v = arena[s.off:s.off + s.size].view(s.rows, s.ld)[:, :s.cols]
        if key == "encoder.0.weight":
            return v.t()                                   # [h0, N] as nn.Linear stores it
        return v[0] if s.vec else v

    def export(self, arena: torch.Tensor):
        return {k: self.view(arena, k).detach().clone().contiguous() for k in self.reference_keys()}

    def load(self, arena: torch.Tensor, sd, prefix=""):
        with torch.no_grad():
            for k in self.reference_keys():
                src = sd[prefix + k]
                dst = self.view(arena, k)
                if tuple(src.shape) != tuple(dst.shape):
                    raise RuntimeError(f"size mismatch for {k}: checkpoint {tuple(src.shape)} vs model {tuple(dst.shape)}")
                dst.copy_(src)


class Workspace:
    """Grow-only device buffers keyed by name."""

    def __init__(self, device):
        self.device, self.buf = device, {}
        self.generation = 0      # bumped whenever a buffer is (re)allocated: captured CUDA graphs hold raw pointers

    def get(self, name, shape, dtype=torch.float32, zero=False, fill=None):
        n = int(np.prod(shape)) if len(shape) else 1
        t = self.buf.get(name)
        if t is None or t.numel() < n or t.dtype != dtype:
            t = torch.empty(max(n, 1), dtype=dtype, device=self.device)
            if zero:
                t.zero_()
            if fill is not None:
                t.fill_(fill)
            self.buf[name] = t
            self.generation += 1
        return t[:n].view(*shape) if len(shape) else t[:1]


class Batch:
    """A batch of users: rows (device int32 or None = 0..B-1) into a device CSR."""

    def __init__(self, csr, rows, B, nnz_cap, b_global=None, nnz_cap_global=None):
        self.csr, self.rows, self.B, self.nnz_cap = csr, rows, B, nnz_cap
        # data-parallel steps: size of the global batch this is a slice of, and the nnz bound of that global batch
        self.b_global, self.nnz_cap_global = b_global, nnz_cap_global


class DeviceCSR:
    """User x item interactions resident in HBM: indptr int64, indices int32, values f32 (or None = ones)."""

    def __init__(self, indptr, indices, values, n_users, n_items, host_lengths=None):
        self.indptr, self.indices, self.values = indptr, indices, values
        self.n_users, self.n_items = n_users, n_items
        self.host_lengths = host_lengths  # numpy int64 [U], for batch nnz caps without a device sync

    @staticmethod
    def from_scipy(m, device, keep_values=None):
        m = m.tocsr()
        if not m.has_sorted_indices:
            m = m.copy()
            m.sort_indices()
        vals = np.asarray(m.data, dtype=np.float32)
        if keep_values is None:
            keep_values = not np.all(vals == 1.0)
        return DeviceCSR(torch.from_numpy(np.asarray(m.indptr, dtype=np.int64)).to(device),
                         torch.from_numpy(np.asarray(m.indices, dtype=np.int32)).to(device),
                         torch.from_numpy(vals).to(device) if keep_values else None,
                         m.shape[0], m.shape[1], np.diff(m.indptr).astype(np.int64))

    @staticmethod
    def from_arrays(indptr, indices, values, n_items, device):
        indptr = np.asarray(indptr, dtype=np.int64)
        return DeviceCSR(torch.from_numpy(indptr).to(device), torch.from_numpy(np.asarray(indices, dtype=np.int32)).to(device),
                         None if values is None else torch.from_numpy(np.asarray(values, dtype=np.float32)).to(device),
                         indptr.shape[0] - 1, n_items, np.diff(indptr))

    @staticmethod
    def from_dense(x: torch.Tensor):
        """Dense [B,N] float rows -> CSR on the device (every non-zero counts, negatives included:
        the reference's tests feed randn, tests/test_unit.py:153-172)."""
        nz = x != 0
        counts = nz.sum(dim=1, dtype=torch.int64)
        indptr = torch.zeros(x.shape[0] + 1, dtype=torch.int64, device=x.device)
        torch.cumsum(counts, 0, out=indptr[1:])
        r, c = torch.nonzero(nz, as_tuple=True)
        return DeviceCSR(indptr, c.to(torch.int32), x[r, c].to(torch.float32).contiguous(), x.shape[0], x.shape[1],
                         counts.cpu().numpy())

    def full_batch(self):
        return Batch(self, None, self.n_users, max(1, int(self.host_lengths.sum())))

    def batch(self, rows_dev, rows_host=None, nnz_cap=None):
        B = rows_dev.shape[0]
        if nnz_cap is None:
            nnz_cap = int(self.host_lengths[rows_host].sum()) if rows_host is not None else int(self.host_lengths.sum())
        return Batch(self, rows_dev, B, max(1, nnz_cap))


class _Span:
    """CUDA-event pair around a named kernel group on the launching stream (bench / profiling only)."""

    def __init__(self, eng, name):
        self.eng, self.name = eng, name

    def __enter__(self):
        if self.eng.prof is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.a.record(torch.cuda.current_stream(self.eng.dev))

    def __exit__(self, *exc):
        if self.eng.prof is not None:
            self.b.record(torch.cuda.current_stream(self.eng.dev))
            self.eng.prof.setdefault(self.name, []).append((self.a, self.b))


class Engine:
    ADAM_B1, ADAM_B2, ADAM_EPS, MAX_NORM = 0.9, 0.999, 1e-8, 5.0
    FUSE_DEFAULT = 0      # measured (profiles/r02_ncu_summary.md section 7): every fusion lengthens the captured step

    def __init__(self, layout: Layout, arena: torch.Tensor, E: torch.Tensor, dropout: float, precision: str = "fp32"):
        if not arena.is_cuda:
            raise RuntimeError("hvae_b200 runs on CUDA devices only (there is no CPU fallback); move the model with .to('cuda')")
        self.lay, self.arena, self.E = layout, arena, E
        self.dropout, self.precision = float(dropout), precision
        self.keep_scale = 1.0 / (1.0 - self.dropout) if self.dropout < 1.0 else 0.0
        self.dev = arena.device
        self.ws = Workspace(self.dev)
        self.lib = _cabi.lib()
        self.state = torch.zeros(STATE_WORDS, dtype=torch.float32, device=self.dev)
        self.m = self.v = self.gd = None
        self.acc = torch.zeros(4, dtype=torch.float32, device=self.dev)     # epoch loss accumulators
        self.loss_out = torch.zeros(3, dtype=torch.float32, device=self.dev)
        self.slot_of_item = None
        self.dist = None  # set by hvae_b200.dist for data-parallel training
        self._E_bf16 = None
        # bf16 mode: GELU/dropout, the bf16 cast of u, the latent backward and the bias-gradient column sums ride in GEMM epilogues
        # HVAE_FUSE: bit mask of the fusions (1 GELU+dropout forward, 2 bf16 copy of u, 4 GELU backward, 8 latent backward, 16 bias-gradient
        # column sums inside those epilogues, 32 one-pass split combination inside du_finalize)
        self.fuse = 0 if precision == "fp32" else int(os.environ.get("HVAE_FUSE", str(self.FUSE_DEFAULT)))
        self.ub_fresh = None
        self._loss_pending = None
        self.adam_split = os.environ.get("HVAE_ADAM_SPLIT", "1") != "0"
        self.two_pass = os.environ.get("HVAE_TWO_PASS", "0") == "1"   # bf16 training: forward-LSE + backward launches instead of the one-pass kernel
        self.prof = None  # dict name -> [(start, stop) events] when profiling spans are enabled
        self.concurrent, self._side, self._forked = False, [], set()

    def span(self, name):
        return _Span(self, name)

    # -- concurrency inside a captured step: independent kernels go to side streams (fork/join edges of the CUDA graph)
    def side(self, i):
        """Context manager: run the enclosed launches on side stream i, ordered after everything enqueued so far on
        the main stream.  Only active while `self.concurrent` (set by the trainer around graph capture)."""
        if not self.concurrent:
            return contextlib.nullcontext()
        while len(self._side) <= i:
            # stream 7 carries the bulk Adam traffic beside the backward pass: lowest priority, so that the (small, latency-bound) kernels
            # of every other branch get SM slots as soon as they are ready instead of queueing behind its half a million blocks
            self._side.append(torch.cuda.Stream(self.dev, priority=0 if len(self._side) == 7 else -1))
        st = self._side[i]
        st.wait_stream(torch.cuda.current_stream(self.dev))
        self._forked.add(i)
        return torch.cuda.stream(st)

    def join(self, only=None, skip=()):
        """Main stream waits for every side stream used since the last join (or just for the streams in `only`; never for `skip`)."""
        if self._forked:
            cur = torch.cuda.current_stream(self.dev)
            for i in sorted((self._forked if only is None else self._forked & set(only)) - set(skip)):
                cur.wait_stream(self._side[i])
                self._forked.discard(i)

    def span_ms(self):
        """{name: [ms per occurrence]} of the recorded spans (synchronises)."""
        torch.cuda.synchronize(self.dev)
        return {k: [a.elapsed_time(b) for a, b in v] for k, v in (self.prof or {}).items()}

    @property
    def E_bf16(self):
        """bf16 copy [N, r8(d)] (zero-padded columns) of the frozen item matrix for the tensor-core scoring
        kernels: half the HBM bytes, rows 16-byte aligned for TMA."""
        if self._E_bf16 is None:
            N, d = self.lay.N, self.lay.d
            self._E_bf16 = torch.empty(N, r8(d), dtype=torch.bfloat16, device=self.dev)
            self.lib.cast_bf16(p(self.E), N, d, d, p(self._E_bf16), r8(d), self.stream)
        return self._E_bf16

    def invalidate_embeddings(self):
        self._E_bf16 = None

    # -- helpers -----------------------------------------------------------------------------------------
    @property
    def stream(self):
        return torch.cuda.current_stream(self.dev).cuda_stream

    def P(self, key):
        """Device pointer of a parameter slot inside the arena."""
        if key in ("fc_mu.bias",):
            key = "fc_ml.bias"
        return self.arena.data_ptr() + 4 * self.lay.slots[key].off

    def G(self, key):
        """Device pointer of a dense-gradient slot (gd is laid out like the arena minus W1^T)."""
        if key in ("fc_mu.bias",):
            key = "fc_ml.bias"
        return self.gd.data_ptr() + 4 * (self.lay.slots[key].off - self.lay.n_w1)

    def read_state(self):
        """Host copy of the step scalars (device->host sync; tests and logging only)."""
        raw = self.state.cpu().numpy()
        out = {k: float(raw[o]) for k, o in STATE_OFF.items()}
        out["adam_step"], out["anneal_step"] = int(raw[:2].view(np.int32)[0]), int(raw[:2].view(np.int32)[1])
        return out

    def state_ptr(self, field):
        return self.state.data_ptr() + 4 * STATE_OFF[field]

    def ensure_optimizer(self):
        if self.m is None:
            self.m = torch.zeros_like(self.arena)
            self.v = torch.zeros_like(self.arena)
        if self.gd is None:
            self.gd = torch.zeros(self.lay.n_dense, dtype=torch.float32, device=self.dev)
        if self.slot_of_item is None:
            self.slot_of_item = torch.full((self.lay.N,), -1, dtype=torch.int32, device=self.dev)

    def gemm(self, M, N, K, A, a_rs, a_cs, Bp, b_rs, b_cs, C, ldc, bias=None, alpha=1.0):
        """fp32 FFMA GEMM (exact mode; materialised scores in either mode)."""
        self.lib.gemm_f32(M, N, K, A, a_rs, a_cs, Bp, b_rs, b_cs, C, ldc, bias, alpha, self.stream)

    def mm(self, M, N, K, A, a_rs, a_cs, Bp, b_rs, b_cs, C, ldc, bias=None, alpha=1.0):
        """GEMM of the MLP stack: tensor cores (TF32 operands, fp32 accumulation) in bf16 mode, FFMA in fp32 mode."""
        if self.precision != "fp32" and self.lib.gemm_tf32_supported(A, a_rs, a_cs, Bp, b_rs, b_cs):
            self.lib.gemm_tf32(M, N, K, A, a_rs, a_cs, Bp, b_rs, b_cs, C, ldc, bias, alpha, self.stream)
        else:
            self.lib.gemm_f32(M, N, K, A, a_rs, a_cs, Bp, b_rs, b_cs, C, ldc, bias, alpha, self.stream)

    # -- forward ---------------------------------------------------------------------------------------------
    def encode(self, batch: Batch, masks=None, keep=True):
        """Encoder up to [mu | logvar].  Returns the `ml` buffer view [B, 2L(+pad)]."""
        lay, ws, lib, st = self.lay, self.ws, self.lib, self.stream
        B, h = batch.B, lay.hidden
        csr = batch.csr
        acts = []
        for i, hi in enumerate(h):
            ld = r4(hi)
            pre = ws.get(f"pre{i}", (B, ld))
            act = ws.get(f"act{i}", (B, ld))
            mean, rstd = ws.get(f"mean{i}", (B,)), ws.get(f"rstd{i}", (B,))
            mask = None if masks is None else masks[i]
            if i == 0:
                with self.span("gather"):
                    lib.gather_ln_fwd(p(csr.indptr), p(csr.indices), p(csr.values), p(batch.rows), B, self.P("encoder.0.weight"),
                                      ld, hi, self.P("encoder.0.bias"), self.P("encoder.1.weight"), self.P("encoder.1.bias"),
                                      p(mask), self.keep_scale, p(pre), p(mean), p(rstd), p(act), st)
            else:
                w = lay.slots[f"encoder.{4 * i}.weight"]
                self.mm(B, hi, h[i - 1], p(acts[-1]), r4(h[i - 1]), 1, self.P(f"encoder.{4 * i}.weight"), 1, w.ld,
                          p(pre), ld, self.P(f"encoder.{4 * i}.bias"))
                lib.ln_act_fwd(p(pre), B, hi, ld, self.P(f"encoder.{4 * i + 1}.weight"), self.P(f"encoder.{4 * i + 1}.bias"),
                               p(mask), self.keep_scale, p(mean), p(rstd), p(act), st)
            acts.append(act)
        L = lay.L
        ldml = r4(2 * L)
        ml = ws.get("ml", (B, ldml))
        wm = lay.slots["fc_mu.weight"]
        self.mm(B, 2 * L, h[-1], p(acts[-1]), r4(h[-1]), 1, self.P("fc_mu.weight"), 1, wm.ld, p(ml), ldml, self.P("fc_ml.bias"))
        return ml

    def latent_and_project(self, B, ml, eps=None, pmask=None, want_kl=True):
        """z = mu (+ eps*std), KL rows, then the projection MLP (or identity) -> u [B, ld(d)]."""
        lay, ws, lib, st = self.lay, self.ws, self.lib, self.stream
        L, d = lay.L, lay.d
        ldml, ldz, ldd = r4(2 * L), r4(L), r4(d)
        z = ws.get("z", (B, ldz))
        kl_row = ws.get("kl_row", (B,))
        lib.reparam_kl(p(ml), ldml, p(eps), B, L, p(z), ldz, p(kl_row) if want_kl else None, st)
        if lay.identity_proj:
            return z
        q, t, u = ws.get("q", (B, ldd)), ws.get("t", (B, ldd)), ws.get("u", (B, ldd))
        w0, w3 = lay.slots["projection_layer.0.weight"], lay.slots["projection_layer.3.weight"]
        if self.fuse & 1:        # GELU + dropout in the epilogue of the GEMM
            lib.gemm_tf32_gelu_drop(B, d, L, p(z), ldz, 1, self.P("projection_layer.0.weight"), 1, w0.ld, p(q), p(t), ldd,
                                    self.P("projection_layer.0.bias"), p(pmask), self.keep_scale, st)
        else:
            self.mm(B, d, L, p(z), ldz, 1, self.P("projection_layer.0.weight"), 1, w0.ld, p(q), ldd, self.P("projection_layer.0.bias"))
            lib.gelu_drop_fwd(p(q), p(pmask), self.keep_scale, B, d, ldd, p(t), st)
        if self.fuse & 2:        # the bf16 copy of u (operand of the scoring kernels) written by the epilogue
            ub = ws.get("u_bf16", (B, r8(d)), torch.bfloat16)
            lib.gemm_tf32_bf16(B, d, d, p(t), ldd, 1, self.P("projection_layer.3.weight"), 1, w3.ld, p(u), ldd,
                               self.P("projection_layer.3.bias"), p(ub), r8(d), st)
            self.ub_fresh = (u.data_ptr(), B)        # consumed (once) by tc.user_vectors_bf16
        else:
            self.mm(B, d, d, p(t), ldd, 1, self.P("projection_layer.3.weight"), 1, w3.ld, p(u), ldd, self.P("projection_layer.3.bias"))
        return u

    def scores_dense(self, u, B, out=None):
        """Materialised S = u E^T [B, N] fp32 (decode(), src/ml/model.py:198)."""
        lay = self.lay
        S = out if out is not None else torch.empty(B, lay.N, dtype=torch.float32, device=self.dev)
        self.gemm(B, lay.N, lay.d, p(u), r4(lay.d), 1, p(self.E), 1, lay.d, p(S), lay.N)
        return S

    def _chunk_rows(self, B):
        budget = 256 * 1024 * 1024  # floats per score chunk (1 GiB)
        return max(1, min(B, budget // max(1, self.lay.N)))

    def score_loss_fp32(self, batch: Batch, u, want_grad: bool):
        """Exact mode: chunked materialised scores -> lse (and O = softmax*|x|/Bg . E when training)."""
        lay, ws, lib, st = self.lay, self.ws, self.lib, self.stream
        B, N, d, ldd = batch.B, lay.N, lay.d, r4(lay.d)
        csr = batch.csr
        lse, dot, xsum = ws.get("lse", (B,)), ws.get("dot", (B,)), ws.get("xsum", (B,))
        lib.sparse_dot_xsum(p(csr.indptr), p(csr.indices), p(csr.values), p(batch.rows), B, p(u), ldd, p(self.E), d, d, 0,
                            p(dot), p(xsum), st)
        O = ws.get("O", (B, ldd)) if want_grad else None
        bc = self._chunk_rows(B)
        S = ws.get("S", (bc, N))
        for r0 in range(0, B, bc):
            nb = min(bc, B - r0)
            up = u.data_ptr() + 4 * r0 * ldd
            self.gemm(nb, N, d, up, ldd, 1, p(self.E), 1, d, p(S), N)
            lib.row_lse(p(S), N, nb, N, lse.data_ptr() + 4 * r0, st)
            if want_grad:
                lib.row_softmax_scale(p(S), N, nb, N, lse.data_ptr() + 4 * r0, xsum.data_ptr() + 4 * r0, self.state_ptr("inv_bg"), st)
                self.gemm(nb, d, N, p(S), N, 1, p(self.E), d, 1, O.data_ptr() + 4 * r0 * ldd, ldd)
        return lse, dot, xsum, O, None

    def score_loss(self, batch, u, want_grad):
        if self.precision == "fp32":
            return self.score_loss_fp32(batch, u, want_grad)
        from . import tc
        return tc.score_loss_bf16(self, batch, u, want_grad)

    # -- one full training step ---------------------------------------------------------------------------------
    def begin(self, b_global, lr=1e-3, beta_min=0.0, beta_max=0.2, anneal_steps=0, advance=True, noise_stride=0):
        self.lib.step_begin(p(self.state), lr, self.ADAM_B1, self.ADAM_B2, beta_min, beta_max, anneal_steps, b_global,
                            1 if advance else 0, int(noise_stride), self.stream)

    def forward_loss(self, batch: Batch, noise=None, want_grad=False, accumulate=True):
        """Forward + loss.  noise = dict(masks=[uint8 [B,h_i]...], eps=f32 [B,L], pmask=uint8 [B,d]) or None."""
        masks = None if noise is None else noise["masks"]
        self.join(only=(3,))            # hidden-layer dropout masks (generated on a side stream by the trainer)
        ml = self.encode(batch, masks)
        self.join(only=(4, 5))          # eps, projection dropout mask
        u = self.latent_and_project(batch.B, ml, None if noise is None else noise["eps"],
                                    None if noise is None else noise.get("pmask"))
        with self.span("score"):
            lse, dot, xsum, O, oscale = self.score_loss(batch, u, want_grad)
        self.join()

        def finalize():
            with self.side(1):          # nothing downstream of the loss scalars inside the step: off the critical path
                self.lib.loss_finalize(p(lse), p(dot), p(xsum), p(self.ws.get("kl_row", (batch.B,))), batch.B, self.state_ptr("inv_bg"),
                                       self.state_ptr("beta_kl"), p(self.loss_out), p(self.acc) if accumulate else None, self.stream)
        if isinstance(oscale, tuple) and len(oscale) == 3:
            self._loss_pending = finalize       # lse comes out of du_finalize_onepass (first kernel of backward())
        else:
            finalize()
        return ml, u, O, oscale

    def backward(self, batch: Batch, noise, ml, O, oscale, dense_w1=None, ext_dml=None, du_override=None):
        """Backward of the loss into self.gd (dense tensors) and the compact layer-1 gradient (or dense_w1)."""
        lay, ws, lib, st = self.lay, self.ws, self.lib, self.stream
        B, L, d, h = batch.B, lay.L, lay.d, lay.hidden
        ldml, ldz, ldd = r4(2 * L), r4(L), r4(d)
        csr = batch.csr
        masks = None if noise is None else noise["masks"]
        eps = None if noise is None else noise["eps"]
        pmask = None if noise is None else noise.get("pmask")
        cs_ws = ws.get("colsum_ws", (64 * max(max(h), 2 * L, d) + 64,))     # side stream 1 only
        cs_ws2 = cs_ws                                                      # (same stream -> same scratch is safe)
        fuse = self.fuse if ext_dml is None else 0
        f_gelu, f_lat, f_cs = bool(fuse & 4), bool(fuse & 8) and not lay.identity_proj, bool(fuse & 16)
        if du_override is not None:
            dU = du_override
        else:
            dU = ws.get("dU", (B, ldd))
            is_bf16 = 0 if self.precision == "fp32" else 1
            Eg, lde = (self.E, d) if not is_bf16 else (self.E_bf16, r8(d))
            n_parts = O.shape[0] if O.dim() == 3 else 1
            if isinstance(oscale, tuple) and len(oscale) == 3:       # one-pass scoring: the split combination rides in this kernel
                oscale, (c_part, l_part, n_sub), lse = oscale
                lib.du_finalize_onepass(p(csr.indptr), p(csr.indices), p(csr.values), p(batch.rows), B, p(O), ldd, n_parts, p(oscale),
                                        p(c_part), p(l_part), n_sub, p(lse), p(Eg), lde, d, is_bf16, self.state_ptr("inv_bg"), p(dU), ldd, st)
                self._loss_pending()
                self._loss_pending = None
            else:
                oscale, w_part = oscale if isinstance(oscale, tuple) else (oscale, None)
                lib.du_finalize(p(csr.indptr), p(csr.indices), p(csr.values), p(batch.rows), B, p(O), ldd, n_parts, p(oscale), p(w_part),
                                p(Eg), lde, d, is_bf16, self.state_ptr("inv_bg"), p(dU), ldd, st)
        if lay.identity_proj:
            dz = dU
        else:
            q, t, z = ws.get("q", (B, ldd)), ws.get("t", (B, ldd)), ws.get("z", (B, ldz))
            w0, w3 = lay.slots["projection_layer.0.weight"], lay.slots["projection_layer.3.weight"]
            # dWp3 = dU^T t ; dbp3 = colsum(dU) ; dt = dU Wp3   (three independent kernels: side streams 0/1 + main)
            with self.side(0):
                self.mm(d, d, B, p(dU), 1, ldd, p(t), ldd, 1, self.G("projection_layer.3.weight"), w3.ld)
            with self.side(1):
                lib.colsum(p(dU), ldd, B, d, self.G("projection_layer.3.bias"), p(cs_ws), self.stream)
            dq = ws.get("dq", (B, ldd))
            if f_gelu:
                # dq = (dU Wp3) * dropout * gelu'(q) (and its column sums = d bias of projection_layer.0) in one launch
                lib.gemm_tf32_gelu_bwd(B, d, d, p(dU), ldd, 1, self.P("projection_layer.3.weight"), w3.ld, 1, p(dq), ldd, p(q), p(pmask),
                                       self.keep_scale, self.G("projection_layer.0.bias") if f_cs else None,
                                       p(self._colsum_ws("dq", B, d)) if f_cs else None, st)
            else:
                dt = ws.get("dt", (B, ldd))
                self.mm(B, d, d, p(dU), ldd, 1, self.P("projection_layer.3.weight"), w3.ld, 1, p(dt), ldd)
                lib.gelu_drop_bwd(p(dt), p(q), p(pmask), self.keep_scale, B, d, ldd, p(dq), st)
            if not (f_gelu and f_cs):
                with self.side(1):
                    lib.colsum(p(dq), ldd, B, d, self.G("projection_layer.0.bias"), p(cs_ws2), self.stream)
            with self.side(0):
                self.mm(d, L, B, p(dq), 1, ldd, p(z), ldz, 1, self.G("projection_layer.0.weight"), w0.ld)
            if not f_lat:
                dz = ws.get("dz", (B, ldz))
                self.mm(B, L, d, p(dq), ldd, 1, self.P("projection_layer.0.weight"), w0.ld, 1, p(dz), ldz)
        dml = ws.get("dml", (B, ldml))
        if f_lat:
            # dz = dq Wp0 never leaves the chip: the epilogue turns it into [dmu | dlogvar] (+ KL gradient) (and sums the columns)
            lib.gemm_tf32_latent_bwd(B, L, d, p(dq), ldd, 1, self.P("projection_layer.0.weight"), w0.ld, 1, p(ml), ldml, p(eps),
                                     self.state_ptr("kl_coef"), p(dml), self.G("fc_ml.bias") if f_cs else None,
                                     p(self._colsum_ws("dml", B, 2 * L)) if f_cs else None, st)
        else:
            lib.latent_bwd(p(dz), ldz, p(ml), ldml, p(eps), B, L, self.state_ptr("kl_coef") if ext_dml is None else p(self._zero()),
                           p(dml), st)
        if ext_dml is not None:
            dml[:, :2 * L].add_(ext_dml)
        wm = lay.slots["fc_mu.weight"]
        nh = len(h)
        act_last = ws.get(f"act{nh - 1}", (B, r4(h[-1])))
        with self.side(0):
            self.mm(2 * L, h[-1], B, p(dml), 1, ldml, p(act_last), r4(h[-1]), 1, self.G("fc_mu.weight"), wm.ld)
        if not (f_lat and f_cs):
            with self.side(1):
                lib.colsum(p(dml), ldml, B, 2 * L, self.G("fc_ml.bias"), p(cs_ws), self.stream)
        if self.dist is not None and dense_w1 is None:      # data parallel: these gradients are complete -> all-reduce them now, on the side
            self.dist.reduce_dense_early(self)
        dact = ws.get(f"dact{nh - 1}", (B, r4(h[-1])))
        self.mm(B, h[-1], 2 * L, p(dml), ldml, 1, self.P("fc_mu.weight"), wm.ld, 1, p(dact), r4(h[-1]))
        ln_ws = ws.get("ln_ws", (max(lib.ln_bwd_workspace_floats(B, r4(hh)) for hh in h),))
        for i in range(nh - 1, -1, -1):
            hi, ld = h[i], r4(h[i])
            pre, mean, rstd = ws.get(f"pre{i}", (B, ld)), ws.get(f"mean{i}", (B,)), ws.get(f"rstd{i}", (B,))
            gk, bk = (f"encoder.{4 * i + 1}.weight", f"encoder.{4 * i + 1}.bias")
            lib.ln_act_bwd(p(dact), p(pre), p(mean), p(rstd), self.P(gk), self.P(bk), p(None if masks is None else masks[i]),
                           self.keep_scale, B, hi, ld, p(dact), self.G(gk), self.G(bk), p(ln_ws), st)   # dact becomes dpre
            if B > 74 * 8:
                lib.launches += 1                # (large batches: the partial d(gamma), d(beta) rows are summed in two launches)
            with self.side(1):
                lib.colsum(p(dact), ld, B, hi, self.G(f"encoder.{4 * i}.bias"), p(cs_ws), self.stream)
            if i > 0:
                w = lay.slots[f"encoder.{4 * i}.weight"]
                prev = ws.get(f"act{i - 1}", (B, r4(h[i - 1])))
                with self.side(0):
                    self.mm(hi, h[i - 1], B, p(dact), 1, ld, p(prev), r4(h[i - 1]), 1, self.G(f"encoder.{4 * i}.weight"), w.ld)
                dprev = ws.get(f"dact{i - 1}", (B, r4(h[i - 1])))
                self.mm(B, h[i - 1], hi, p(dact), ld, 1, self.P(f"encoder.{4 * i}.weight"), w.ld, 1, p(dprev), r4(h[i - 1]))
                dact = dprev
        self.dpre0 = dact
        if dense_w1 is not None:
            lib.w1_grad_dense(p(csr.indptr), p(csr.indices), p(csr.values), p(batch.rows), B, p(dact), r4(h[0]), h[0], p(dense_w1), st)

    def _colsum_ws(self, name, B, cols):
        """Zero-initialised workspace of the column sums a fused GEMM epilogue produces (the kernel leaves its counters zero)."""
        return self.ws.get("gemm_colsum_" + name, (int(self.lib.gemm_colsum_workspace_floats(B, cols)),), zero=True)

    def _zero(self):
        return self.ws.get("zero1", (1,), zero=True)

    def transpose_batch(self, batch: Batch):
        """Sort the batch's (user, item, value) entries by item (stable): segment s = the entries of touched item s.
        Depends on the batch only, so a captured step runs it beside the forward pass."""
        lay, ws, lib, st = self.lay, self.ws, self.lib, self.stream
        B = batch.B
        csr, cap = batch.csr, batch.nnz_cap
        i32 = torch.int32
        boff = ws.get("boff", (B + 1,), i32)
        names = ["keys", "keys_sorted", "eid", "eid_sorted", "head", "slot", "ent_user", "uniq_item"]
        arr = {n: ws.get("bt_" + n, (cap,), i32) for n in names}
        ent_val = ws.get("bt_ent_val", (cap,))
        seg_start = ws.get("bt_seg_start", (cap + 1,), i32)
        n_unique = ws.get("bt_n_unique", (1,), i32, zero=True)
        overflow = ws.get("bt_overflow", (1,), i32, zero=True)
        tb = int(lib.batch_temp_bytes(cap, lay.N))
        temp = ws.get("bt_temp", (tb,), torch.uint8)
        lib.batch_offsets(p(csr.indptr), p(batch.rows), B, p(boff), st)
        lib.batch_transpose(p(csr.indptr), p(csr.indices), p(csr.values), p(batch.rows), B, lay.N, cap, p(boff), p(arr["keys"]),
                            p(arr["keys_sorted"]), p(arr["eid"]), p(arr["eid_sorted"]), p(arr["head"]), p(arr["slot"]),
                            p(arr["ent_user"]), p(ent_val), p(seg_start), p(arr["uniq_item"]), p(self.slot_of_item), p(n_unique),
                            p(overflow), p(temp), tb, st)
        chunk_base = ws.get("w1_chunk_base", (cap + 1,), i32)
        part_base = ws.get("w1_part_base", (cap + 1,), i32)
        work_slot = ws.get("w1_work_slot", (int(lib.w1_max_work(cap)),), i32)
        multi_slot = ws.get("w1_multi_slot", (int(lib.w1_max_partial_rows(cap)),), i32)
        n_work = ws.get("w1_n_work", (2,), i32, zero=True)
        lib.w1_plan(p(seg_start), p(n_unique), cap, p(chunk_base), p(part_base), p(work_slot), p(multi_slot), p(n_work), st)
        return dict(cap=cap, overflow=overflow, seg_start=seg_start, n_unique=n_unique, eid_sorted=arr["eid_sorted"], ent_user=arr["ent_user"],
                    ent_val=ent_val, uniq=arr["uniq_item"], chunk_base=chunk_base, part_base=part_base, work_slot=work_slot,
                    multi_slot=multi_slot, n_work=n_work)

    def w1_grad(self, tb, dpre_ptr, block_rows=0, block_stride=0):
        """d(W1^T) rows of the touched items (deterministic segment sums) and their squared norms.  dpre_ptr: device
        pointer of the batch's d(pre-activation) rows (optionally blocked: see hvae_w1_grad)."""
        ws, lib = self.ws, self.lib
        ld1 = r4(self.lay.hidden[0])
        n_rows = min(tb["cap"], self.lay.N)            # at most one gradient row per item
        gs = ws.get("gs", (n_rows, ld1))
        rn2 = ws.get("rownorm2", (tb["cap"],))
        part = ws.get("w1_partial", (int(lib.w1_max_partial_rows(tb["cap"])), ld1))
        lib.w1_grad(p(tb["seg_start"]), p(tb["n_unique"]), p(tb["eid_sorted"]), p(tb["ent_user"]), p(tb["ent_val"]), tb["cap"],
                    p(tb["chunk_base"]), p(tb["part_base"]), p(tb["work_slot"]), p(tb["multi_slot"]), p(tb["n_work"]), dpre_ptr, ld1, block_rows,
                    block_stride, p(gs), p(part), p(rn2), self.stream)
        return gs, rn2

    def sparse_w1_grad(self, batch: Batch, dpre0, B=None):
        """Transpose the batch by item and reduce d(W1^T) rows (deterministic)."""
        tb = self.transpose_batch(batch)
        gs, rn2 = self.w1_grad(tb, p(dpre0))
        return gs, rn2, tb["n_unique"], tb["uniq"]

    def train_step(self, batch: Batch, noise, lr=1e-3, weight_decay=0.0, beta_min=0.0, beta_max=0.2, anneal_steps=0,
                   b_global=None, noise_stride=0, begun=False):
        """zero_grad + forward + loss + backward + clip_grad_norm_(5) + Adam (src/ml/train.py:88-92), fused."""
        self.ensure_optimizer()
        lib, st, lay = self.lib, self.stream, self.lay
        b_global = batch.B if b_global is None else b_global
        self.b_global = b_global
        if not begun:      # (the trainer calls begin() itself before it forks the noise kernels onto side streams)
            self.begin(b_global, lr, beta_min, beta_max, anneal_steps, advance=True, noise_stride=noise_stride)
        # the item-major view of the (global) batch does not depend on the forward pass: side stream
        with self.side(2), self.span("transpose"):
            wbatch = batch if self.dist is None else self.dist.gather_batch(self, batch)
            tb = self.transpose_batch(wbatch)
        ml, u, O, oscale = self.forward_loss(batch, noise, want_grad=True)
        if self.adam_split:
            # Adam for the W1^T rows WITHOUT a gradient in this step (most of them: moments decay, the row moves along its momentum) needs
            # nothing from the backward pass: its 24 B/parameter stream runs on a side stream beside the latency-bound backward kernels
            # (NOT beside the scoring kernel: measured, that one loses more L2 bandwidth than the overlap gains)
            with self.side(7), self.span("adam_untouched"):
                if self.concurrent and len(self._side) > 2:
                    torch.cuda.current_stream(self.dev).wait_stream(self._side[2])        # slot_of_item comes from the transposition
                lib.adam_step_untouched(p(self.arena), p(self.m), p(self.v), lay.n_w1, r4(lay.hidden[0]), p(self.slot_of_item), p(self.state),
                                        weight_decay, self.ADAM_B1, self.ADAM_B2, self.ADAM_EPS, self.stream)
        with self.span("bwd_dense"):
            self.backward(batch, noise, ml, O, oscale)
        self.join(skip=(7,))
        dpre_ptr, block_rows, block_stride = p(self.dpre0), 0, 0
        if self.dist is not None:
            with self.span("exchange"):
                dpre_ptr, block_rows, block_stride = self.dist.exchange_grads(self, batch, self.dpre0)
        gn_ws = self.ws.get("gn_ws", (256,))
        with self.side(1):           # the dense gradients are final: their sum of squares runs beside the layer-1 gradient kernels
            lib.grad_sumsq_dense(p(self.gd), lay.n_dense, p(gn_ws), self.stream)
        with self.span("w1grad"):
            gs, rn2 = self.w1_grad(tb, dpre_ptr, block_rows, block_stride)
        n_unique, uniq = tb["n_unique"], tb["uniq"]
        self.join(only=(1,))
        lib.grad_norm_finish(lay.n_dense, p(rn2), p(n_unique), self.MAX_NORM, p(self.state), p(gn_ws), st)
        with self.span("adam"):
            if self.adam_split:
                self.join(only=(7,))
                lib.adam_step_touched(p(self.arena), p(self.m), p(self.v), lay.n_params, lay.n_w1, r4(lay.hidden[0]), p(uniq), p(n_unique),
                                      min(tb["cap"], lay.N), p(gs), p(self.gd), p(self.state), weight_decay, self.ADAM_B1, self.ADAM_B2,
                                      self.ADAM_EPS, st)
            else:
                lib.adam_step(p(self.arena), p(self.m), p(self.v), lay.n_params, lay.n_w1, r4(lay.hidden[0]), p(self.slot_of_item), p(gs),
                              p(self.gd), p(self.state), weight_decay, self.ADAM_B1, self.ADAM_B2, self.ADAM_EPS, st)
        # restores slot_of_item; a batch that did not fit its nnz bound turns the step's loss into NaN (see check_overflow)
        lib.batch_release(p(uniq), p(n_unique), wbatch.nnz_cap, p(self.slot_of_item), p(tb["overflow"]), p(self.loss_out), p(self.acc), st)

    def check_overflow(self):
        """Raise if a training step since the last call dropped batch rows because its nnz bound (Batch.nnz_cap /
        nnz_cap_global) was too small -- such a step has an incomplete layer-1 weight gradient.  Called by the trainer
        whenever it reads a NaN loss back (the kernels poison the loss of such a step), so it costs nothing per step."""
        ov = self.ws.buf.get("bt_overflow")
        if ov is not None and int(ov[0].item()) != 0:
            n = int(ov[0].item())
            ov.zero_()
            raise RuntimeError(f"hvae_b200: {n} batch row(s) did not fit the batch's nnz bound (Batch.nnz_cap / nnz_cap_global too "
                               "small): the layer-1 weight gradient of that step was incomplete; pass an exact bound")

    def eval_step(self, batch: Batch, beta, b_global=None):
        """Validation forward: eval mode (z = mu, no dropout), fixed beta (src/ml/train.py:105-117)."""
        self.begin(batch.B if b_global is None else b_global, beta_max=beta, anneal_steps=0, advance=False)
        self.forward_loss(batch, None, want_grad=False)

    # -- scoring / top-K -----------------------------------------------------------------------------------------
    def user_vectors(self, batch: Batch):
        """u = projection(mu) for a batch in eval mode (get_user_embedding + decode prologue)."""
        ml = self.encode(batch, None)
        return self.latent_and_project(batch.B, ml, None, None, want_kl=False)

    def topk(self, batch: Batch, K: int, exclude_seen=True, item_lo=0, item_hi=None, *, mask=None, allow=None):
        """Full ranking: scores over items [item_lo,item_hi) -> mask seen -> top-K (value, global index).

        mask = (indptr int64 [B+1], indices int32): sorted items to leave out per batch row, used instead of the seen rows
        (exclude_seen is then not looked at).  allow = (bitmaps int32 [F, words], allow_of_row int32 [B]): item allow-sets
        over global ids, -1 = unrestricted.  Slots a filtered row cannot fill hold (-inf, -1)."""
        lay, ws, lib, st = self.lay, self.ws, self.lib, self.stream
        item_hi = lay.N if item_hi is None else item_hi
        n_it = item_hi - item_lo
        B, d, ldd = batch.B, lay.d, r4(lay.d)
        u = self.user_vectors(batch)
        out_val = torch.empty(B, K, dtype=torch.float32, device=self.dev)
        out_idx = torch.empty(B, K, dtype=torch.int32, device=self.dev)
        if self.precision != "fp32":
            from . import tc
            if tc.topk_bf16(self, batch, u, K, exclude_seen, item_lo, item_hi, out_val, out_idx, mask, allow):
                return out_val, out_idx
        csr = batch.csr
        bc = max(1, min(B, (256 * 1024 * 1024) // max(1, n_it)))
        S = ws.get("S", (bc, n_it))
        rows = batch.rows if batch.rows is not None else torch.arange(B, dtype=torch.int32, device=self.dev)
        for r0 in range(0, B, bc):
            nb = min(bc, B - r0)
            self.gemm(nb, n_it, d, u.data_ptr() + 4 * r0 * ldd, ldd, 1, self.E.data_ptr() + 4 * item_lo * d, 1, d, p(S), n_it)
            rows_ptr = rows.data_ptr() + 4 * r0
            nc = int(lib.mask_topk_chunks(nb, n_it))
            cv = ws.get("topk_cand_v", (nb, nc * K))
            ci = ws.get("topk_cand_i", (nb, nc * K), torch.int32)
            ov, oi = out_val.data_ptr() + 4 * r0 * K, out_idx.data_ptr() + 4 * r0 * K
            if mask is None and allow is None:
                lib.mask_topk(p(S), n_it, nb, n_it, item_lo, p(csr.indptr), p(csr.indices), rows_ptr, 1 if exclude_seen else 0, K,
                              p(cv), p(ci), ov, oi, st)
                continue
            if mask is not None:        # rows of the mask CSR are batch rows: start at row r0 of it
                indptr_ptr, indices_ptr, rows_ptr, excl = mask[0].data_ptr() + 8 * r0, p(mask[1]), None, 1
            else:
                indptr_ptr, indices_ptr, excl = p(csr.indptr), p(csr.indices), 1 if exclude_seen else 0
            bm, aor = allow if allow is not None else (None, None)
            lib.mask_topk_filtered(p(S), n_it, nb, n_it, item_lo, indptr_ptr, indices_ptr, rows_ptr, excl, p(bm),
                                   0 if bm is None else bm.stride(0), None if aor is None else aor.data_ptr() + 4 * r0, K,
                                   p(cv), p(ci), ov, oi, st)
        return out_val, out_idx
