"""Board power and SM clock while the fused contraction runs back to back for ~2 s.  Shows what the launch costs in a
burst vs sustained."""
import os, sys, subprocess, statistics, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "pytorch-nmf_b200")]
import torch
from torchnmf_b200.engine import CudaNmfEngine, release_workspaces
prec = sys.argv[1] if len(sys.argv) > 1 else "f16"
N, C, R = 65536, 4096, 64
torch.manual_seed(0)
V = torch.rand(N, C, device="cuda").bfloat16().float()
W = torch.randn(C, R, device="cuda").abs(); H = torch.randn(N, R, device="cuda").abs()
eng = CudaNmfEngine(V, W, H, prec)
for _ in range(5): eng.contract_only(1, 1.0)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(10): eng.contract_only(1, 1.0)
e1.record(); torch.cuda.synchronize()
burst = e0.elapsed_time(e1) / 10 * 1e3
time.sleep(1.0)
smi = subprocess.Popen(["nvidia-smi", "--query-gpu=power.draw,clocks.sm", "--format=csv,noheader,nounits", "-lms", "50"],
                       stdout=subprocess.PIPE, text=True)
n = int(2.0e6 / burst)
e0.record()
for _ in range(n): eng.contract_only(1, 1.0)
e1.record(); torch.cuda.synchronize()
sus = e0.elapsed_time(e1) / n * 1e3
smi.terminate()
rows = [l.split(",") for l in smi.stdout.read().strip().splitlines() if "," in l]
pw = sorted(float(r[0]) for r in rows); ck = sorted(float(r[1]) for r in rows)
top = pw[len(pw) // 2:]                       # samples taken under load (the first ones still ramp)
print(f"full kernel  burst {burst:6.1f} us  sustained {sus:6.1f} us  power {statistics.median(top):5.0f} W  "
      f"clock {statistics.median(ck[:len(ck) // 2 + 1]):5.0f} MHz ({len(rows)} samples)", flush=True)
eng.close(); release_workspaces()
