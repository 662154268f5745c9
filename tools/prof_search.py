"""Profiling target: build an N x 384 index and run a few searches (for ncu / variant timing)."""
import os, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ragmeup_b200.index import FlatIndex, MODE_AUTO, MODE_TENSOR_NOFALLBACK
MODE = MODE_TENSOR_NOFALLBACK if os.environ.get('RMU_SEARCH_NOFALLBACK') == '1' else MODE_AUTO
N = int(os.environ.get("PROF_N", 10_000_000)); Q = int(os.environ.get("PROF_Q", 128)); K = int(os.environ.get("PROF_K", 10)); D = int(os.environ.get("PROF_D", 384))
IT = int(os.environ.get("PROF_ITERS", 3)); metric = os.environ.get("PROF_METRIC", "ip")
dev = torch.device("cuda")
def unit(n, d, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    return torch.nn.functional.normalize(torch.randn(n, d, generator=g, device=dev), dim=1)
ix = FlatIndex(D, metric); ix.reserve(N)
for b in range(0, N, 1_000_000):
    ix.add(unit(min(1_000_000, N - b), D, 100 + b // 1_000_000))
qs = unit(Q, D, 5)
torch.cuda.synchronize()
ts = []
for it in range(IT):
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(); ix.search(qs, K, mode=MODE); e1.record(); torch.cuda.synchronize()
    ts.append(e0.elapsed_time(e1))
print(f"N={N} Q={Q} k={K} {metric}: ms per search {['%.3f' % t for t in ts]}  "
      f"{4.0*N*D/(min(ts)*1e-3)/1e9:.0f} GB/s D={D}", flush=True)
if os.environ.get("PROF_CLASSES") == "1":
    from ragmeup_b200 import _lib
    _lib.profile_enable(True); _lib.profile_reset()
    for _ in range(10): ix.search(qs, K, mode=MODE)
    torch.cuda.synchronize()
    print({k: (round(v[0] / 10, 4), v[1] // 10) for k, v in _lib.profile_read().items() if v[1]}, flush=True)
    _lib.profile_enable(False)
