import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "pytorch-nmf_b200")]
import torch
from torchnmf_b200.engine import CudaNmfEngine
prec, N, C, reps = sys.argv[1], int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4])
R = 64
torch.manual_seed(0)
V = torch.rand(N, C, device="cuda").bfloat16().float()
W = torch.randn(C, R, device="cuda").abs(); H = torch.randn(N, R, device="cuda").abs()
eng = CudaNmfEngine(V, W, H, prec)
t0 = time.time()
try:
    for i in range(reps):
        eng.contract_only(i & 1, 1.0)
        if i % 200 == 199:
            eng.check_health()
    eng.check_health()
    print(f"OK   {prec} N={N} C={C} {reps} launches {time.time()-t0:.2f}s", flush=True)
except Exception as e:
    print(f"FAIL {prec} N={N} C={C} after {time.time()-t0:.3f}s: {str(e)[:80]}", flush=True)
