import sys
from pathlib import Path
ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / "recommendation-system_b200")]
import torch
from hvae_b200 import _cabi
lib=_cabi.lib()
torch.zeros(1,device='cuda')
for smem in (199168, 215040, 224*1024, 229376+1024, 231424, 232448-1024, 232448):
    print(smem, lib.tc_duo_max_clusters(smem), lib._dll.hvae_last_error().decode() if lib.tc_duo_max_clusters(smem)<0 else '')
print(torch.cuda.get_device_properties(0))
