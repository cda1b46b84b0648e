"""bench.py -- MU iterations/sec of the dense NMF hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N --steps K --warmup W] [--impl reference|reference-cuda]
                    [--config cfg2|cfg1|cfg3|cfg4s|cfg5] [--beta B] [--precision auto|f32|f16|f16_split]
                    [--dump-outputs DIR]

A "step" is one `fit(V, beta, tol=-inf, max_iter=ITERS)` pass (the reference's own benchmark protocol,
examples/benchmarks/benchmark.ipynb cell 4: loss evaluations every 10 iterations included) on one
synthetic batch: V = rand(N, C) rounded to bf16-representable values, W0/H0 = |randn| (SURVEY 8d).

  value : ITERS * K * n_gpus / t   with V, W, H resident in HBM (one shard per GPU)
  e2e   : the same through the public API with HOST (pinned) tensors: the module and V live on the CPU,
          `fit` stages V/W/H through the GPU and copies the factors back, all inside the timed region
  roofline / cpu_baseline / gpu_reference : see DESIGN.md section "Measurement"

Configs (BASELINE.json `configs`): cfg1 256x512 R=16 beta=2 | cfg2 65536x4096 R=64 KL (the metric's config, default) |
cfg3 NMFD 1025x8192 R=16 T=128 KL | cfg4s one 131072x8192 R=128 row shard (1/8) of the 8192 x 2^20 problem |
cfg5 = cfg2's shape with --beta in {0, 0.5, 1, 1.5, 2}.

Multi-GPU (torchrun): rows are sharded, W is replicated, one all-reduce per W update; weak scaling (every rank owns a
full shard), value = shard-iterations of all ranks per second.  The main line stays on the metric's config (cfg2
shards); every multi-GPU line (and the N=1 line) also carries `north_star_cfg4` = the same measurement on the
131072x8192 R=128 shards of BASELINE.json configs[3] (N=8 is exactly that problem) and, for N>1, `sharded_check` = a
200-iteration sharded fit compared with the single-rank fit of the concatenated problem.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "pytorch-nmf_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402

CONFIGS = {
    # name: (kind, shape, beta, description)   NMF shape = (N, C, R); NMFD shape = (B, C, L, R, T)
    "cfg1": ("nmf", (256, 512, 16), 2.0, "NMF 256x512 rank=16 beta=2 (BASELINE.json configs[0])"),
    "cfg2": ("nmf", (65536, 4096, 64), 1.0,
             "NMF 4096x65536 (fed as V^T: 65536x4096) rank=64 beta=1 KL (BASELINE.json configs[1])"),
    "cfg3": ("nmfd", (1, 1025, 8192, 16, 128), 1.0,
             "NMFD spectrogram 1025x8192 R=16 T=128 beta=1 (BASELINE.json configs[2])"),
    "cfg4s": ("nmf", (131072, 8192, 128), 1.0,
              "one 1/8 row shard (131072x8192) of NMF 8192x2^20 rank=128 beta=1 (BASELINE.json configs[3])"),
    "cfg5": ("nmf", (65536, 4096, 64), None,
             "beta sweep on 4096x65536 (fed as 65536x4096) rank=64, one beta per run (BASELINE.json configs[4])"),
}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tc=d["bf16_tflops"], tc_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tc=1590.0, tc_sustained=1400.0, src="fallback")


def ncu_traffic(precision, cfg_name):
    """(bytes, source file): dram read+write bytes per launch of the fused contraction kernel from the newest committed
    `ncu --set full` capture of this precision at cfg2.  It is a replayed constant, not measured in this run."""
    if cfg_name not in ("cfg2", "cfg5"):
        return None, None
    for rnd in ("r2", "r1"):
        rel = os.path.join("profiles", f"{rnd}_ncu_tc_contract_{precision}.txt")
        try:
            tot, launches = 0.0, 0
            for ln in open(os.path.join(ROOT, rel)):
                ln = ln.strip()
                if ln.startswith("dram__bytes_read.sum") or ln.startswith("dram__bytes_write.sum"):
                    val, unit = ln.split("=")[1].split()[:2]
                    tot += float(val) * {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}[unit]
                    launches += ln.startswith("dram__bytes_read.sum")
            if tot:
                return tot / max(launches, 1), rel      # the capture may hold the W and the H launch: per-launch mean
        except Exception:
            continue
    return None, None


def make_inputs(N, C, R, seed, floor=0.0):
    torch.manual_seed(seed)
    V = torch.rand(N, C).bfloat16().float()
    if floor > 0:
        V.clamp_(min=floor)
    torch.manual_seed(seed + 1)
    W0 = torch.randn(C, R).abs()
    H0 = torch.randn(N, R).abs()
    return V, W0, H0


def make_inputs_nmfd(B, C, L, R, T, seed):
    torch.manual_seed(seed)
    V = torch.rand(B, C, L).bfloat16().float()
    torch.manual_seed(seed + 1)
    W0 = torch.randn(C, R, T).abs()
    H0 = torch.randn(B, R, L - T + 1).abs()
    return V, W0, H0


def v_floor(beta):
    return 2.0 ** -7 if beta <= 0 else 0.0       # nmf.py:332-336: beta <= 0 needs a strictly positive target


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def wait_ready(self, timeout=0.5):
        """Block (briefly) until nvidia-smi has delivered its first line."""
        t0 = time.time()
        while self.proc and not self.lines and time.time() - t0 < timeout:
            time.sleep(0.01)

    def mark(self):
        """The timed region starts now: only samples that arrive from here on are reported (nvidia-smi takes ~0.1 s to come up,
        so it is started one warm-up step early and a short timed region would otherwise end before its first line)."""
        self.first = len(self.lines)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, watts = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        first = getattr(self, "first", 0)
        window = "timed region"
        if len(self.lines) <= first and self.lines:      # region shorter than one sampling period: the warm-up step before it
            first, window = 0, "last warm-up step + timed region"
        self.window = window
        for ln in self.lines[first:]:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); smax = float(f[1])
            except ValueError:
                continue
            try:
                watts.append(float(f[2]))
            except ValueError:
                pass
            for nm, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        top = sm[len(sm) // 2:] if sm else []        # samples under load = upper half
        med = top[len(top) // 2] if top else None
        watts.sort()
        wtop = watts[len(watts) // 2:] if watts else []     # board power under load (DESIGN.md 4.1: the cfg2 line sits at the cap)
        return {"sm_mhz": med, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm), "window": self.window,
                "board_power_w": wtop[len(wtop) // 2] if wtop else None}


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write what the timed path returned as <out_dir>/<name>.npy in float32, so that two builds can be compared output
    for output.  Past DUMP_BYTES in all, the largest array keeps a fixed, seeded sample of its rows (sorted)."""
    import numpy as np
    host = {k: v.detach().float().cpu() for k, v in arrays.items()}
    total = sum(t.numel() * 4 for t in host.values())
    if total > DUMP_BYTES:
        k = max(host, key=lambda n: host[n].numel())
        t = host[k]
        rows = (DUMP_BYTES - (total - t.numel() * 4)) // (t[0].numel() * 4)
        idx = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:rows].sort().values
        host[k] = t[idx]
    os.makedirs(out_dir, exist_ok=True)
    for k, t in host.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), t.numpy())


def dist_setup(n_gpus):
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local


def timed_steps(fn, steps, warmup, world):
    """W warm-up steps, then exactly K timed steps bracketed by barrier + synchronize; device time, max over ranks."""
    import torch.distributed as dist
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    ev[0].record()
    for i in range(steps):
        fn()
        ev[i + 1].record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[-1])
    timed_steps.per_step = [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]
    if world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms


def reference_module():
    """The unmodified reference (baseline/_ref, pip-installed from /root/reference) or None."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    if os.path.isdir(os.path.join(ref, "torchnmf")):
        if ref not in sys.path:
            sys.path.insert(0, ref)
        import torchnmf.nmf as rn
        return rn
    return None


def cpu_reference_rate(kind, V, W0, H0, beta, iters, warm=True):
    """it/s of the reference's CPU path: one discarded fit(max_iter=1), then fit(tol=-inf, max_iter=iters) timed
    (BASELINE.md section 4) on all host cores.  Falls back to the oracle port when baseline/_ref is absent."""
    torch.set_num_threads(os.cpu_count())
    try:
        torch.set_flush_denormal(True)       # README.md:101-102 of the reference
    except Exception:
        pass
    rn = reference_module()
    if rn is not None:
        cls = rn.NMF if kind == "nmf" else rn.NMFD
        label = "reference"
        if warm:
            cls(W=W0, H=H0).fit(V, beta, float("-inf"), 1)
        m = cls(W=W0, H=H0)
        t0 = time.perf_counter()
        n = m.fit(V, beta, float("-inf"), iters)
        dt = time.perf_counter() - t0
    else:
        from oracle import mu_oracle as orc
        label = "port"
        if warm:
            orc.fit(V, W0, H0, beta=beta, tol=float("-inf"), max_iter=1, kind=kind)
        t0 = time.perf_counter()
        _, _, n, _ = orc.fit(V, W0, H0, beta=beta, tol=float("-inf"), max_iter=iters, kind=kind)
        dt = time.perf_counter() - t0
    return n / dt, label, torch.get_num_threads(), dt


def gpu_reference_rate(kind, V_dev, W0, H0, beta, iters):
    """it/s of the UNMODIFIED reference moved to the same B200 with .cuda() (cuBLAS + unfused ATen ops, fp32, the two
    autograd backward passes of nmf.py:52-92): the "library path on the same box" line (BASELINE.md section 4)."""
    rn = reference_module()
    if rn is None:
        return None
    cls = rn.NMF if kind == "nmf" else rn.NMFD
    try:
        m = cls(W=W0, H=H0).cuda()
        m.fit(V_dev, beta, float("-inf"), 2)
        torch.cuda.synchronize()
        m = cls(W=W0, H=H0).cuda()
        t0 = time.perf_counter()
        n = m.fit(V_dev, beta, float("-inf"), iters)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        del m
        torch.cuda.empty_cache()
        return {"value": n / dt, "unit": "iter/s", "kind": "reference torchnmf 0.3.5 .cuda() fp32 on this GPU (stock code path)",
                "sample": f"fit(tol=-inf, max_iter={iters}) after a 2-iteration warm-up, same target"}
    except Exception as e:          # e.g. out of memory for the materialised WH temporaries
        torch.cuda.empty_cache()
        return {"value": None, "unavailable": f"{type(e).__name__}: {str(e)[:120]}"}


def config_inputs(cfg_name, beta, seed):
    kind, shape, _, _ = CONFIGS[cfg_name]
    if kind == "nmf":
        N, C, R = shape
        return make_inputs(N, C, R, seed, v_floor(beta))
    return make_inputs_nmfd(*shape, seed)


def run_reference_arm(a, cfg_name, beta):
    """`--impl reference`: the reference's own CPU implementation (baseline/_ref) on this box's host cores, rank 0 only.
    Same protocol as the `cpu_baseline` of the main arm: a discarded 1-iteration fit, then K x fit(max_iter=ref_iters)."""
    kind, shape, _, desc = CONFIGS[cfg_name]
    if int(os.environ.get("RANK", "0")) != 0:
        return
    V, W0, H0 = config_inputs(cfg_name, beta, 0)
    it = a.ref_iters
    cpu_reference_rate(kind, V, W0, H0, beta, 1, warm=False)            # warm-up (first-call cost)
    for _ in range(max(0, a.warmup - 1)):
        cpu_reference_rate(kind, V, W0, H0, beta, 1, warm=False)
    t0 = time.perf_counter()
    label, cores = "port", 1
    for _ in range(a.steps):
        _, label, cores, _ = cpu_reference_rate(kind, V, W0, H0, beta, it, warm=False)
    dt = time.perf_counter() - t0
    rate = a.steps * it / dt
    line = {
        "impl": "reference", "metric": "MU iterations/sec", "value": rate, "unit": "iter/s", "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * dt / a.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(cfg_name, beta, 1, it, "f32"),
        "cpu_baseline": {"value": rate, "unit": "iter/s", "cores": cores, "kind": label,
                         "sample": f"{a.steps} x fit(tol=-inf, max_iter={it}) on the full target {tuple(V.shape)} after "
                                   "1-iteration warm-up fits (each fit includes its init loss evaluation)"},
        "e2e": {"value": rate, "unit": "iter/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def run_reference_cuda_arm(a, cfg_name, beta):
    """`--impl reference-cuda`: the unmodified reference on the GPU (.cuda()), same metric / config."""
    kind, shape, _, desc = CONFIGS[cfg_name]
    if int(os.environ.get("RANK", "0")) != 0:
        return
    V, W0, H0 = config_inputs(cfg_name, beta, 0)
    V_dev = V.cuda()
    res = None
    t0 = time.perf_counter()
    for _ in range(a.steps):
        res = gpu_reference_rate(kind, V_dev, W0, H0, beta, a.iters)
    dt = time.perf_counter() - t0
    if not res or res.get("value") is None:
        emit({"impl": "reference-cuda", "unavailable": (res or {}).get("unavailable", "baseline/_ref not installed")})
        return
    emit({"impl": "reference-cuda", "metric": "MU iterations/sec", "value": res["value"], "unit": "iter/s", "n_gpus": 1,
          "steps": a.steps, "warmup": 1, "ms_per_step": 1e3 * dt / a.steps, "higher_is_better": True, "scaling": "weak",
          "vs_baseline": None, "dtype": "f32", "data": "synthetic",
          "config": workload_config(cfg_name, beta, 1, a.iters, "f32"), "gpu_reference": res, "gpu_launches": 0})


def workload_config(cfg_name, beta, world, iters, precision):
    kind, shape, _, desc = CONFIGS[cfg_name]
    c = {"workload": desc, "beta": beta, "iters_per_step": iters, "precision": precision,
         "unit_def": "one MU iteration (W then H update) over one per-GPU shard; loss every 10th iteration included",
         "parallelism": f"row-shard x{world}" if world > 1 else "single"}
    if kind == "nmf":
        N, C, R = shape
        c.update({"N_per_gpu": N, "C": C, "R": R,
                  "l2": "inputs larger than L2 (V shard >= 512 MiB)" if N * C * 2 > 126e6 else "inputs fit in L2"})
    else:
        B, C, L, R, T = shape
        c.update({"B": B, "C": C, "L": L, "R": R, "T": T,
                  "l2": "inputs fit in L2 (V 33.6 MB): the path is compute-bound; every iteration rewrites the ratio "
                        "matrix, nothing is cached between steps"})
    return c


_REAL_STDOUT = None


def _capture_stdout():
    """Everything libraries print to fd 1 (e.g. NCCL's version banner) goes to stderr; the one JSON line is written
    to the real stdout by emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def flops_per_iter(kind, shape, beta):
    """Algorithmic FLOPs of one MU iteration of the algorithm actually run (SURVEY 8d)."""
    if kind == "nmfd":
        B, C, L, R, T = shape
        return 4 * 2.0 * B * C * R * T * (L - T + 1) * (1.0 if beta == 1 else 1.5)
    N, C, R = shape
    if beta == 1:
        return 8.0 * N * C * R
    if beta == 2:
        return 4.0 * N * C * R        # residual tile + Gram-matrix denominators: one contraction pair per factor
    return 12.0 * N * C * R


def sharded_check(dev, rank, world, group, precision):
    """200 KL iterations of a 4096x1024 R=64 problem, row-sharded over `world` ranks, against the single-rank fit of the
    concatenated problem (run redundantly on every rank): W replicas must be bit-identical, W and H within rtol 1e-3."""
    import torch.distributed as dist
    from torchnmf_b200 import NMF
    N, C, R, iters = 4096, 1024, 64, 200
    V, W0, H0 = make_inputs(N, C, R, 100)
    rows = N // world
    lo, hi = rank * rows, (rank + 1) * rows if rank < world - 1 else N
    ms = NMF(W=W0, H=H0[lo:hi]).to(dev)
    n = ms.fit(V[lo:hi].to(dev), 1, float("-inf"), iters, precision=precision, group=group)
    full = NMF(W=W0, H=H0).to(dev)
    full.fit(V.to(dev), 1, float("-inf"), iters, precision=precision)
    Ws = [torch.empty_like(ms.W.data) for _ in range(world)]
    dist.all_gather(Ws, ms.W.data.contiguous(), group=group)
    identical = all(torch.equal(Ws[0], w) for w in Ws[1:])

    def rel(a, b):
        atol = 1e-5 * float(b.abs().max())
        return float(((a - b).abs() / (b.abs() * 1e-3 + atol)).max())       # in units of the tolerance (rtol 1e-3)

    e = torch.tensor([rel(ms.W.data, full.W.data), rel(ms.H.data, full.H.data[lo:hi])], device=dev, dtype=torch.float64)
    dist.all_reduce(e, op=dist.ReduceOp.MAX, group=group)
    err = float(e.max())
    return {"ok": bool(identical and err <= 1.0 and n == iters), "w_replicas_identical": bool(identical),
            "max_err_over_tol": err, "tol": "rtol 1e-3, atol 1e-5*max", "case": f"{N}x{C} R={R} KL {iters} it, "
            f"{world} row shards vs the single-rank fit", "precision": ms.last_fit_precision,
            "w_update_path": ms.last_w_update_path}


def cfg4_shard_rate(dev, rank, world, group, precision, iters=40):
    """Device-resident it/s on the 131072x8192 R=128 row shards of BASELINE.json configs[3] (inputs generated on the
    GPU, seed = rank; W replicas start identical).  Returns the per-rank iteration rate (max time over ranks)."""
    import torch.distributed as dist
    from torchnmf_b200 import NMF
    N, C, R = CONFIGS["cfg4s"][1]
    g = torch.Generator(device=dev); g.manual_seed(1000 + rank)
    V = torch.rand(N, C, device=dev, generator=g).bfloat16().float()
    H0 = torch.randn(N, R, device=dev, generator=g).abs()
    g.manual_seed(7)
    W0 = torch.randn(C, R, device=dev, generator=g).abs()
    m = NMF((N, C), R)
    m = m.to(dev)
    m.W.data.copy_(W0); m.H.data.copy_(H0)

    def step():
        m.W.data.copy_(W0); m.H.data.copy_(H0)
        n = m.fit(V, 1, float("-inf"), iters, precision=precision, group=group)
        assert n == iters

    ms = timed_steps(step, 2, 2, world)
    rate = iters * 2 / (ms * 1e-3)
    fl = flops_per_iter("nmf", (N, C, R), 1.0)
    peaks = load_peaks()
    out = {"workload": CONFIGS["cfg4s"][3], "iters_per_s_per_rank": rate, "shard_iters_per_s": rate * world,
           "n_gpus": world, "ms_per_iter": 1e3 / rate, "precision": m.last_fit_precision,
           "tensor_frac_of_sustained_peak": fl * rate / 1e12 / peaks["tc_sustained"],
           "note": "N = 8 is exactly the 8192 x 2^20 problem; at N < 8 every rank still owns one 131072-row shard (weak scaling)"}
    del m, V, H0
    torch.cuda.empty_cache()
    return out


def main():
    _capture_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-cuda"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--beta", type=float, default=None, help="cfg5: the beta of this run (0, 0.5, 1, 1.5, 2)")
    ap.add_argument("--iters", type=int, default=None, help="MU iterations per step (fit max_iter)")
    ap.add_argument("--ref-iters", type=int, default=5, help="MU iterations per reference step")
    ap.add_argument("--precision", default="auto")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip north_star_cfg4 / sharded_check")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write W and H of the last timed step (rank 0's shard) to DIR/W.npy, DIR/H.npy (float32, <= 64 MB)")
    a = ap.parse_args()
    kind, shape, beta, desc = CONFIGS[a.config]
    if beta is None:
        beta = 1.0 if a.beta is None else a.beta
    elif a.beta is not None:
        beta = a.beta
    if a.iters is None:
        a.iters = 200 if (kind == "nmf" and a.config != "cfg4s") else (40 if a.config == "cfg4s" else 100)
    if a.impl == "reference":
        run_reference_arm(a, a.config, beta)
        return
    if a.impl == "reference-cuda":
        run_reference_cuda_arm(a, a.config, beta)
        return

    assert torch.cuda.is_available(), "bench.py needs a CUDA device"
    rank, world, local = dist_setup(a.gpus)
    assert world == a.gpus, f"--gpus {a.gpus} but WORLD_SIZE={world} (launch N>1 with torch.distributed.run)"
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    import torch.distributed as dist
    from torchnmf_b200 import NMF, NMFD, _capi
    from torchnmf_b200.engine import CudaNmfEngine
    peaks = load_peaks()
    group = dist.group.WORLD if world > 1 else None
    if kind == "nmfd" and world > 1:
        group = None                     # NMFD: replicas only (DESIGN.md section 7)

    # ---------------- inputs: one full shard per rank (weak scaling) -----------------------------------
    V_cpu, W0, H0 = config_inputs(a.config, beta, 2 * rank)
    if world > 1 and kind == "nmf":     # W replicas must start identical
        torch.manual_seed(1)
        W0 = torch.randn(*W0.shape).abs()
    V_cpu = V_cpu.pin_memory()
    V_dev = V_cpu.to(dev)
    cls = NMF if kind == "nmf" else NMFD
    model = cls(W=W0, H=H0).to(dev)
    W0d, H0d = W0.to(dev), H0.to(dev)

    def step_resident():
        model.W.data.copy_(W0d); model.H.data.copy_(H0d)
        n = model.fit(V_dev, beta, float("-inf"), a.iters, precision=a.precision, group=group)
        assert n == a.iters

    sampler = ClockSampler(torch.cuda.current_device()) if rank == 0 else None
    # warm-up, with the sampler brought up during its last step; only the samples of the timed steps are reported
    for i in range(a.warmup):
        if sampler and i == a.warmup - 1:
            sampler.start()
        step_resident()
    torch.cuda.synchronize()
    if sampler:
        if a.warmup == 0:
            sampler.start()
        sampler.wait_ready()          # rank 0 only; the other ranks meet it at the barrier that opens the timed region
        sampler.mark()
    l0 = _capi.launch_count()
    ms = timed_steps(step_resident, a.steps, 0, world)
    launches = _capi.launch_count() - l0
    per_step = list(getattr(timed_steps, "per_step", []))
    clocks = sampler.stop() if sampler else None
    precision = model.last_fit_precision
    value = a.iters * a.steps * world / (ms * 1e-3)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, {"W": model.W.data, "H": model.H.data})

    # ---------------- end to end through the public API with host buffers ------------------------------
    e2e = None
    if not a.no_e2e:
        host_model = cls(W=W0, H=H0)          # CPU-resident module, like the reference's default
        for p in (host_model.W, host_model.H):
            p.data = p.data.pin_memory()
        W0p, H0p = W0.pin_memory(), H0.pin_memory()

        def step_host():
            host_model.W.data.copy_(W0p); host_model.H.data.copy_(H0p)
            n = host_model.fit(V_cpu, beta, float("-inf"), a.iters, precision=a.precision, group=group)
            assert n == a.iters

        for _ in range(max(1, a.warmup // 2)):
            step_host()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            step_host()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        n_loss = 1 + a.iters // 10
        e2e = {"value": a.iters * a.steps * world / dt, "unit": "iter/s",
               "h2d_bytes_per_step": int(V_cpu.nbytes + W0.nbytes + H0.nbytes),
               "d2h_bytes_per_step": int(W0.nbytes + H0.nbytes + 8 * n_loss + 8),
               "ms_per_step": 1e3 * dt / a.steps}

    # ---------------- roofline -------------------------------------------------------------------------------
    fl_iter = flops_per_iter(kind, shape, beta)
    step_tf = fl_iter * a.iters * a.steps / (ms * 1e-3) / 1e12           # per GPU
    if kind == "nmf":
        # dominant kernel = the fused contraction, timed alone with CUDA events on the launching stream
        N, C, R = shape
        eng = CudaNmfEngine(V_dev, model.W.data, model.H.data, a.precision)
        reps = 10
        times = {}
        for which, nm in ((0, "w"), (1, "h")):
            for _ in range(3):
                eng.contract_only(which, beta)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                eng.contract_only(which, beta)
            e1.record()
            torch.cuda.synchronize()
            times[nm] = e0.elapsed_time(e1) / reps * 1e-3
        eng.close()
        flops_launch = fl_iter / 2
        v_bytes = N * C * (4 if precision == "f32" else 2)
        t_dom = max(times.values())
        which_dom = max(times, key=times.get)
        ach_tf = flops_launch / t_dom / 1e12
        ach_gb = v_bytes / t_dom / 1e9
        tensor = {"achieved": ach_tf, "peak": peaks["tc"], "unit": "TFLOP/s", "frac": ach_tf / peaks["tc"],
                  "algorithmic_flops_per_launch": flops_launch,
                  "peak_source": f"{peaks['src']} MEASURED_PEAKS.json bf16 burst (f16 has the same tensor peak)"}
        hbm = {"achieved": ach_gb, "peak": peaks["hbm"], "unit": "GB/s", "frac": ach_gb / peaks["hbm"],
               "algorithmic_bytes_per_launch": v_bytes,
               "peak_source": f"{peaks['src']} MEASURED_PEAKS.json copy bandwidth (burst)"}
        # the binding roofline is the one whose minimum time for this launch is larger (cfg2, R=64: HBM 82 us vs tensor
        # 41 us; at R=128 the two meet); the other one is reported next to it
        hbm_bound = v_bytes / (peaks["hbm"] * 1e9) >= flops_launch / (peaks["tc"] * 1e12) or precision == "f32"
        traffic, traffic_src = ncu_traffic(precision, a.config)
        roof = dict(hbm if hbm_bound else tensor)
        roof.update({"bound": "hbm" if hbm_bound else "tensor", "traffic": traffic, "traffic_source": traffic_src,
                     "kernel": f"fused {which_dom}-update contraction ({precision})", "kernel_ms": t_dom * 1e3,
                     "kernel_ms_w": times["w"] * 1e3, "kernel_ms_h": times["h"] * 1e3,
                     "tensor" if hbm_bound else "hbm": tensor if hbm_bound else hbm,
                     "step_tensor_frac": step_tf / peaks["tc_sustained"],
                     "step_hbm_frac": 2.0 * v_bytes * a.iters * a.steps / (ms * 1e-3) / 1e9 / peaks["hbm"],
                     "algorithmic_flops_per_iteration": fl_iter})
    else:
        roof = {"bound": "tensor", "achieved": step_tf, "peak": peaks["tc_sustained"], "unit": "TFLOP/s",
                "frac": step_tf / peaks["tc_sustained"], "traffic": None, "traffic_source": None,
                "kernel": "NMFD iteration (recon x2, wgrad, dgrad): step-level figure, the target is L2-resident",
                "algorithmic_flops_per_iteration": fl_iter,
                "peak_source": f"{peaks['src']} MEASURED_PEAKS.json bf16 sustained"}

    # ---------------- same-box baselines (rank 0, N=1 only) ------------------------------------------------------
    cpu = gpu_ref = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        cells = V_cpu.numel()
        k = 5 if cells >= 1 << 23 else 50
        rate, label, cores, dt = cpu_reference_rate(kind, V_cpu, W0, H0, beta, k)
        cpu = {"value": rate, "unit": "iter/s", "cores": cores, "kind": label,
               "sample": f"fit(tol=-inf, max_iter={k}) after a 1-iteration warm-up on the full target {tuple(V_cpu.shape)} ({dt:.1f}s)"}
    if rank == 0 and world == 1 and not a.no_gpu_reference:
        gpu_ref = gpu_reference_rate(kind, V_dev, W0, H0, beta, 50 if kind == "nmf" else 20)

    # ---------------- north-star extras: cfg4 shards and the sharded result check ----------------------------------
    extras = {}
    if not a.no_extras and kind == "nmf" and a.config == "cfg2":
        del V_dev
        torch.cuda.empty_cache()
        extras["north_star_cfg4"] = cfg4_shard_rate(dev, rank, world, group, a.precision)
        if world > 1:
            extras["sharded_check"] = sharded_check(dev, rank, world, group, a.precision)

    if rank == 0:
        line = {
            "metric": "MU iterations/sec", "value": value, "unit": "iter/s", "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms / a.steps, "step_ms": per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": {"f32": "f32", "f16": "f16", "f16_split": "f16"}.get(precision, precision),
            "data": "synthetic", "config": dict(workload_config(a.config, beta, world, a.iters, precision),
                                                **({"w_update": "fused P2P sum + ratio stage over NVLink peer memory"
                                                    if getattr(model, "last_w_update_path", None) == "peer" else
                                                    "NCCL all-reduce between contraction and ratio stage"} if world > 1 else {})),
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
            "gpu_reference": gpu_ref,
        }
        line.update(extras)
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
