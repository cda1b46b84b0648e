"""Generate tests/golden/*.npz by running the REAL reference (torchnmf 0.3.5).

TEST INFRASTRUCTURE ONLY (see oracle/mu_oracle.py header).  Run in the build container, where
the reference is importable from /root/reference (read-only) or baseline/_ref:

    python oracle/make_golden.py            # small cases (seconds)
    python oracle/make_golden.py --cfg2     # + the 200-iteration 65536x4096 R=64 KL run (~10 min CPU)

The GPU box has no reference; the fixtures written here are what travels.  Inputs are generated
from fixed torch CPU seeds (SURVEY 8d): V = rand(N,C) rounded to bf16-representable values, so the
fp32 reference and the 16-bit-operand engine consume bit-identical data; W0/H0 = |randn|.  The fixtures store
the reference's outputs and, in place of the inputs, the recipe of oracle/golden_inputs.py that regenerates them
with their sha256 (every file stays under 1 MB).
"""
import argparse
import math
import os
import sys
import time

import numpy as np
import torch

import golden_inputs as gi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for cand in (os.path.join(ROOT, "baseline", "_ref"), "/root/reference"):
    if os.path.isdir(os.path.join(cand, "torchnmf")):
        sys.path.insert(0, cand)
        break
import torchnmf  # noqa: E402  (the reference)
import torchnmf.nmf as ref_nmf  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def make_inputs(shape_v, shape_w, shape_h, seed_v=0, seed_f=1, floor=0.0):
    torch.manual_seed(seed_v)
    V = torch.rand(*shape_v).bfloat16().float()
    if floor > 0:
        V = V.clamp_min(floor)
    torch.manual_seed(seed_f)
    W0 = torch.randn(*shape_w).abs()
    H0 = torch.randn(*shape_h).abs()
    return V, W0, H0


def run_reference(cls, V, W0, H0, beta, tol, max_iter, alpha, l1_ratio, trainable_W=True, trainable_H=True):
    losses = []
    orig = ref_nmf.beta_div

    def recording(inp, tgt, b=2):
        out = orig(inp, tgt, b)
        losses.append(math.sqrt(2.0 * float(out)))
        return out

    ref_nmf.beta_div = recording
    try:
        m = cls(W=W0, H=H0, trainable_W=trainable_W, trainable_H=trainable_H)
        n_iter = m.fit(V, beta, tol, max_iter, False, alpha, l1_ratio)
    finally:
        ref_nmf.beta_div = orig
    return m.W.detach().clone(), m.H.detach().clone(), n_iter, losses


def small_cases():
    torch.set_num_threads(1)          # deterministic MKL reduction order for the fixtures
    cases = {}
    # --- NMF, ragged shape (not a multiple of any tile), all beta branches of nmf.py:61-74 ---
    N, C, R = 97, 83, 8
    for beta in (-1, 0, 0.5, 1, 1.5, 2, 3):
        for alpha, l1r in ((0, 0), (0.1, 0.5)):
            V, W0, H0 = make_inputs((N, C), (C, R), (N, R), floor=2 ** -7 if beta <= 0 else 0.0)
            W, H, n_iter, losses = run_reference(ref_nmf.NMF, V, W0, H0, beta, float("-inf"), 20, alpha, l1r)
            cases[f"nmf_b{beta}_a{alpha}_l{l1r}"] = dict(
                kind="nmf", V=V, W0=W0, H0=H0, W=W, H=H, n_iter=n_iter, losses=losses,
                beta=beta, tol=float("-inf"), max_iter=20, alpha=alpha, l1_ratio=l1r)
    # --- stop rule / trainable flags ---
    V, W0, H0 = make_inputs((N, C), (C, R), (N, R))
    W, H, n_iter, losses = run_reference(ref_nmf.NMF, V, W0, H0, 1, 1e-2, 100, 0, 0)
    cases["nmf_stoprule"] = dict(kind="nmf", V=V, W0=W0, H0=H0, W=W, H=H, n_iter=n_iter, losses=losses,
                                 beta=1, tol=1e-2, max_iter=100, alpha=0, l1_ratio=0)
    W, H, n_iter, losses = run_reference(ref_nmf.NMF, V, W0, H0, 1.5, float("-inf"), 10, 0, 0, trainable_W=False)
    cases["nmf_frozenW"] = dict(kind="nmf", V=V, W0=W0, H0=H0, W=W, H=H, n_iter=n_iter, losses=losses,
                                beta=1.5, tol=float("-inf"), max_iter=10, alpha=0, l1_ratio=0, trainable_W=False)
    # --- BASELINE.json configs[0]: NMF 256x512 rank 16 beta=2, 50 iterations ---
    V, W0, H0 = make_inputs((256, 512), (512, 16), (256, 16))
    W, H, n_iter, losses = run_reference(ref_nmf.NMF, V, W0, H0, 2, float("-inf"), 50, 0, 0)
    cases["nmf_cfg1"] = dict(kind="nmf", V=V, W0=W0, H0=H0, W=W, H=H, n_iter=n_iter, losses=losses,
                             beta=2, tol=float("-inf"), max_iter=50, alpha=0, l1_ratio=0)
    # --- tensor-core-shaped NMF case (R = 64, tile multiples and ragged edges), KL, 30 iterations ---
    for tag, (N2, C2, R2) in (("tc", (384, 256, 64)), ("tcragged", (300, 200, 64))):
        V, W0, H0 = make_inputs((N2, C2), (C2, R2), (N2, R2))
        W, H, n_iter, losses = run_reference(ref_nmf.NMF, V, W0, H0, 1, float("-inf"), 30, 0, 0)
        cases[f"nmf_{tag}"] = dict(kind="nmf", V=V, W0=W0, H0=H0, W=W, H=H, n_iter=n_iter, losses=losses,
                                   beta=1, tol=float("-inf"), max_iter=30, alpha=0, l1_ratio=0)
    # --- NMFD (nmf.py:776-779), batch 2, ragged sizes ---
    B, C, L, R, T = 2, 21, 61, 4, 5
    for beta in (0, 0.5, 1, 2, 3):
        for alpha, l1r in ((0, 0), (0.1, 0.5)):
            V, W0, H0 = make_inputs((B, C, L), (C, R, T), (B, R, L - T + 1), floor=2 ** -7 if beta <= 0 else 0.0)
            W, H, n_iter, losses = run_reference(ref_nmf.NMFD, V, W0, H0, beta, float("-inf"), 20, alpha, l1r)
            cases[f"nmfd_b{beta}_a{alpha}_l{l1r}"] = dict(
                kind="nmfd", V=V, W0=W0, H0=H0, W=W, H=H, n_iter=n_iter, losses=losses,
                beta=beta, tol=float("-inf"), max_iter=20, alpha=alpha, l1_ratio=l1r)
    return cases


def factor_args(V, W0, H0, **kw):
    """Arguments of the `factors` recipe (oracle/golden_inputs.py) that regenerates these make_inputs tensors."""
    return dict(v_shape=list(V.shape), w_shape=list(W0.shape), h_shape=list(H0.shape), **kw)


def save_cases(cases, fname, inputs=None):
    """`inputs(case) -> (recipe, args)` names the recipe of the case's V, W0, H0; by default make_inputs' own, with the
    floor it applies for beta <= 0."""
    flat = {}
    for name, c in cases.items():
        for k, v in c.items():
            if isinstance(v, torch.Tensor):
                v = v.numpy()
            elif k == "kind":
                v = np.array(v)
            elif k == "losses":
                v = np.array(v, dtype=np.float64)
            else:
                v = np.array(v, dtype=np.float64)
            flat[f"{name}/{k}"] = v
        recipe, args = inputs(c) if inputs else (
            "factors", factor_args(c["V"], c["W0"], c["H0"], floor=2 ** -7 if c["beta"] <= 0 else 0.0))
        gi.pack(flat, name, recipe, **args)
    os.makedirs(GOLD, exist_ok=True)
    np.savez_compressed(os.path.join(GOLD, fname), **flat)
    print(f"wrote {fname}: {len(cases)} cases, {os.path.getsize(os.path.join(GOLD, fname)) / 1e6:.2f} MB")


def cfg2_case(iters=200):
    """BASELINE.json configs[1]: V (65536, 4096), R = 64, beta = 1, 200 iterations from seeds 0/1.
    Only subsampled factor rows are stored (W rows ::8, H rows ::128); inputs are regenerated from
    the seeds on the GPU box and verified against the float64 checksums stored here."""
    torch.set_num_threads(os.cpu_count())
    torch.set_flush_denormal(True)     # README.md:101-102
    N, C, R = 65536, 4096, 64
    V, W0, H0 = make_inputs((N, C), (C, R), (N, R))
    t0 = time.time()
    W, H, n_iter, losses = run_reference(ref_nmf.NMF, V, W0, H0, 1, float("-inf"), iters, 0, 0)
    dt = time.time() - t0
    print(f"cfg2 reference: {n_iter} iterations in {dt:.1f}s ({n_iter / dt:.3f} it/s, {os.cpu_count()} threads)")
    np.savez_compressed(
        os.path.join(GOLD, "nmf_cfg2_kl_200.npz"),
        W_sub=W[::8].numpy(), H_sub=H[::128].numpy(), n_iter=np.array(n_iter),
        losses=np.array(losses, dtype=np.float64),
        v_sum=np.array(V.double().sum().item()), w0_sum=np.array(W0.double().sum().item()),
        h0_sum=np.array(H0.double().sum().item()),
        w_absmax=np.array(W.abs().max().item()), h_absmax=np.array(H.abs().max().item()),
        ref_seconds=np.array(dt), ref_threads=np.array(os.cpu_count()), iters=np.array(iters))
    print("wrote nmf_cfg2_kl_200.npz")


# ---------------------------------------------------------------------------------------------------------
# Round 2: goldens at the shapes of BASELINE.json configs[2..4] (kernel paths the small cases never reach).
# Inputs are regenerated from seeds by the tests (checksums stored); only subsampled factors are stored.
# ---------------------------------------------------------------------------------------------------------
def _store(flat, name, V, W0, H0, W, H, n_iter, losses, meta, w_step=1, h_step=1):
    flat[f"{name}/W_sub"] = W[::w_step].numpy()
    flat[f"{name}/H_sub"] = (H[::h_step] if H.dim() == 2 else H[..., ::h_step]).contiguous().numpy()
    flat[f"{name}/w_step"] = np.array(w_step); flat[f"{name}/h_step"] = np.array(h_step)
    flat[f"{name}/n_iter"] = np.array(n_iter)
    flat[f"{name}/losses"] = np.array(losses, dtype=np.float64)
    flat[f"{name}/v_sum"] = np.array(V.double().sum().item())
    flat[f"{name}/w0_sum"] = np.array(W0.double().sum().item())
    flat[f"{name}/h0_sum"] = np.array(H0.double().sum().item())
    flat[f"{name}/w_absmax"] = np.array(W.abs().max().item())
    flat[f"{name}/h_absmax"] = np.array(H.abs().max().item())
    for k, v in meta.items():
        flat[f"{name}/{k}"] = np.array(v, dtype=np.float64)


def heavy_tailed(N, C, seed=0):
    """Spectrogram-like target: lognormal magnitudes over ~6 decades (exercises the fp16 range handling)."""
    torch.manual_seed(seed)
    return torch.exp(2.0 * torch.randn(N, C)).bfloat16().float()


def round2_cases():
    torch.set_num_threads(os.cpu_count())
    torch.set_flush_denormal(True)
    flat = {}
    # --- cfg3: NMFD spectrogram 1025 x 8192, R = 16, T = 128, beta = 1, 20 iterations (reference ~0.8 s / iteration) ---
    t0 = time.time()
    B, C, L, R, T = 1, 1025, 8192, 16, 128
    V, W0, H0 = make_inputs((B, C, L), (C, R, T), (B, R, L - T + 1))
    W, H, n_iter, losses = run_reference(ref_nmf.NMFD, V, W0, H0, 1, float("-inf"), 20, 0, 0)
    _store(flat, "nmfd_cfg3", V, W0, H0, W, H, n_iter, losses,
           dict(B=B, C=C, L=L, R=R, T=T, beta=1, max_iter=20), w_step=64, h_step=8)
    print(f"nmfd_cfg3 {time.time() - t0:.1f}s", flush=True)
    # --- NMFD ragged: T = 37 crosses the 32-wide shift chunk, C = 130 crosses the 128-row tile, batch 2 ---
    B, C, L, R, T = 2, 130, 700, 5, 37
    for beta in (1, 0.5):
        V, W0, H0 = make_inputs((B, C, L), (C, R, T), (B, R, L - T + 1))
        W, H, n_iter, losses = run_reference(ref_nmf.NMFD, V, W0, H0, beta, float("-inf"), 20, 0, 0)
        _store(flat, f"nmfd_ragged_b{beta}", V, W0, H0, W, H, n_iter, losses,
               dict(B=B, C=C, L=L, R=R, T=T, beta=beta, max_iter=20), w_step=2)
    print(f"nmfd_ragged {time.time() - t0:.1f}s", flush=True)
    # --- cfg4-shaped: R = 128 (the 128-column operand kernels), KL, 100 iterations ---
    N, C, R = 8192, 2048, 128
    V, W0, H0 = make_inputs((N, C), (C, R), (N, R))
    W, H, n_iter, losses = run_reference(ref_nmf.NMF, V, W0, H0, 1, float("-inf"), 100, 0, 0)
    _store(flat, "nmf_r128_kl", V, W0, H0, W, H, n_iter, losses, dict(N=N, C=C, R=R, beta=1, max_iter=100), w_step=8, h_step=64)
    print(f"nmf_r128 {time.time() - t0:.1f}s", flush=True)
    # --- cfg5-shaped: beta sweep at R = 64, 50 iterations ---
    N, C, R = 4096, 1024, 64
    for beta in (0, 0.5, 1.5, 2):
        V, W0, H0 = make_inputs((N, C), (C, R), (N, R), floor=2 ** -7 if beta <= 0 else 0.0)
        W, H, n_iter, losses = run_reference(ref_nmf.NMF, V, W0, H0, beta, float("-inf"), 50, 0, 0)
        _store(flat, f"nmf_sweep_b{beta}", V, W0, H0, W, H, n_iter, losses,
               dict(N=N, C=C, R=R, beta=beta, max_iter=50, floor=2 ** -7 if beta <= 0 else 0.0), w_step=16, h_step=64)
    print(f"sweep {time.time() - t0:.1f}s", flush=True)
    # --- heavy-tailed targets (lognormal, ~6 decades): KL and IS, 30 iterations ---
    N, C, R = 1024, 512, 32
    for beta in (1, 0):
        V = heavy_tailed(N, C)
        torch.manual_seed(1)
        W0 = torch.randn(C, R).abs(); H0 = torch.randn(N, R).abs()
        W, H, n_iter, losses = run_reference(ref_nmf.NMF, V, W0, H0, beta, float("-inf"), 30, 0, 0)
        _store(flat, f"nmf_heavy_b{beta}", V, W0, H0, W, H, n_iter, losses,
               dict(N=N, C=C, R=R, beta=beta, max_iter=30), w_step=4, h_step=8)
    np.savez_compressed(os.path.join(GOLD, "reference_r2.npz"), **flat)
    print(f"wrote reference_r2.npz ({os.path.getsize(os.path.join(GOLD, 'reference_r2.npz')) / 1e6:.2f} MB) in {time.time() - t0:.1f}s")


# ---------------------------------------------------------------------------------------------------------
# Round 2, "next" rows: trainer.BetaMu single steps and PLCA fits from the real reference (reference_next.npz)
# ---------------------------------------------------------------------------------------------------------
def next_row_cases():
    import torchnmf.plca as ref_plca
    import torchnmf.trainer as ref_trainer
    torch.set_num_threads(1)
    flat = {}
    # --- BetaMu: three steps over [W, H] of one NMF module, every beta branch, with l1 / l2 / orthogonal penalties ---
    N, C, R = 96, 80, 8
    for beta in (-1, 0, 0.5, 1, 1.5, 2, 3):
        for tag, (l1, l2, ortho) in (("plain", (0, 0, 0)), ("reg", (0.1, 0.05, 0.2))):
            torch.manual_seed(0)
            V = torch.rand(N, C).bfloat16().float() + (2 ** -7 if beta <= 0 else 0.0)
            torch.manual_seed(1)
            W0 = torch.randn(C, R).abs(); H0 = torch.randn(N, R).abs()
            m = ref_nmf.NMF(W=W0, H=H0)
            tr = ref_trainer.BetaMu([m.W, m.H], beta, l1, l2, ortho)

            def closure():
                tr.zero_grad()
                return V, m()
            for _ in range(3):
                tr.step(closure)
            name = f"betamu_b{beta}_{tag}"
            # (the closure's zero_grad() clears W.grad again before H is updated: only the last parameter keeps its .grad)
            for k, v in dict(V=V, W0=W0, H0=H0, W=m.W.detach().clone(), H=m.H.detach().clone(),
                             gH=m.H.grad.clone()).items():
                flat[f"{name}/{k}"] = v.numpy()
            for k, v in dict(beta=beta, l1=l1, l2=l2, ortho=ortho, steps=3).items():
                flat[f"{name}/{k}"] = np.array(v, dtype=np.float64)
            gi.pack(flat, name, "factors", **factor_args(V, W0, H0, offset=2 ** -7 if beta <= 0 else 0.0))
    # --- PLCA: small ragged case (Dirichlet priors, frozen Z) and a tensor-core-shaped case ---
    for name, (N, C, R, iters, kw, fitkw) in {
        "plca_small": (97, 83, 8, 30, {}, {}),
        "plca_prior": (97, 83, 8, 30, {}, dict(W_alpha=1.05, H_alpha=1.02, Z_alpha=1.1)),
        "plca_frozenZ": (97, 83, 8, 20, dict(trainable_Z=False), {}),
        "plca_tc": (1024, 512, 32, 50, {}, {}),
    }.items():
        torch.manual_seed(0)
        V = torch.rand(N, C).bfloat16().float() * 3
        torch.manual_seed(1)
        W0 = torch.randn(C, R).abs(); H0 = torch.randn(N, R).abs(); Z0 = torch.rand(R) + 0.1
        m = ref_plca.PLCA(W=W0, H=H0, Z=Z0, **kw)
        n_iter, norm = m.fit(V, float("-inf"), iters, False, **fitkw)
        for k, v in dict(V=V, W0=W0, H0=H0, Z0=Z0, W=m.W.detach().clone(), H=m.H.detach().clone(),
                         Z=m.Z.detach().clone()).items():
            flat[f"{name}/{k}"] = v.numpy()
        flat[f"{name}/n_iter"] = np.array(n_iter); flat[f"{name}/norm"] = np.array(float(norm)); flat[f"{name}/iters"] = np.array(iters)
        flat[f"{name}/trainable_Z"] = np.array(int(kw.get("trainable_Z", True)))
        for k in ("W_alpha", "H_alpha", "Z_alpha"):
            flat[f"{name}/{k}"] = np.array(float(fitkw.get(k, 1.0)))
        gi.pack(flat, name, "factors", **factor_args(V, W0, H0, scale=3, z=True))
    np.savez_compressed(os.path.join(GOLD, "reference_next.npz"), **flat)
    print(f"wrote reference_next.npz ({os.path.getsize(os.path.join(GOLD, 'reference_next.npz')) / 1e6:.2f} MB)")


# PLCA family: the shift-invariant models through the real reference (reference_plca.npz)
# ---------------------------------------------------------------------------------------------------------
def plca_cases():
    import torchnmf.plca as ref_plca
    torch.set_num_threads(1)
    flat = {}
    #      name              class      V shape              R   kernel      iters  ctor kw                    fit kw
    cases = {
        "siplca_small":    ("SIPLCA",  (2, 21, 61),          5, (6,),       30, {}, {}),
        "siplca_prior":    ("SIPLCA",  (2, 21, 61),          5, (6,),       30, {}, dict(W_alpha=1.0005, H_alpha=1.0002, Z_alpha=1.1)),
        "siplca_sparse":   ("SIPLCA",  (2, 21, 61),          5, (6,),       30, {}, dict(W_alpha=0.9995, H_alpha=0.9995, Z_alpha=0.95)),
        "siplca_frozenZ":  ("SIPLCA",  (1, 21, 61),          5, (6,),       20, dict(trainable_Z=False), {}),
        "siplca_frozenW":  ("SIPLCA",  (1, 21, 61),          5, (6,),       20, dict(trainable_W=False), {}),
        "siplca_onlyH":    ("SIPLCA",  (1, 21, 61),          5, (6,),       20, dict(trainable_W=False, trainable_Z=False), {}),
        "siplca_stop":     ("SIPLCA",  (1, 21, 61),          5, (6,),       200, {}, dict(tol=1e-2)),
        "siplca_tc":       ("SIPLCA",  (1, 257, 1024),       16, (32,),     30, {}, {}),
        "siplca2_small":   ("SIPLCA2", (2, 3, 24, 31),       4, (4, 5),     20, {}, {}),
        "siplca2_prior":   ("SIPLCA2", (1, 3, 24, 31),       4, (4, 5),     20, {}, dict(W_alpha=1.001, H_alpha=1.0005, Z_alpha=1.05)),
        "siplca3_small":   ("SIPLCA3", (1, 2, 10, 12, 14),   3, (2, 3, 4),  15, {}, {}),
    }
    for name, (cls, vshape, R, K, iters, kw, fitkw) in cases.items():
        B, C, *X = vshape
        torch.manual_seed(0)
        V = torch.rand(*vshape).bfloat16().float() * 3
        torch.manual_seed(1)
        W0 = torch.randn(C, R, *K).abs(); H0 = torch.randn(B, R, *(x - k + 1 for x, k in zip(X, K))).abs(); Z0 = torch.rand(R) + 0.1
        m = getattr(ref_plca, cls)(W=W0, H=H0, Z=Z0, **kw)
        fitkw = dict(fitkw)
        tol = fitkw.pop("tol", float("-inf"))
        n_iter, norm = m.fit(V, tol, iters, False, **fitkw)
        for k, v in dict(V=V, W0=W0, H0=H0, Z0=Z0, W=m.W.detach().clone(), H=m.H.detach().clone(),
                         Z=m.Z.detach().clone()).items():
            flat[f"{name}/{k}"] = v.numpy()
        flat[f"{name}/n_iter"] = np.array(n_iter); flat[f"{name}/norm"] = np.array(float(norm)); flat[f"{name}/iters"] = np.array(iters)
        flat[f"{name}/tol"] = np.array(tol, dtype=np.float64)
        flat[f"{name}/cls"] = np.array(int(cls[-1]) if cls[-1].isdigit() else 1)
        for k in ("trainable_W", "trainable_H", "trainable_Z"):
            flat[f"{name}/{k}"] = np.array(int(kw.get(k, True)))
        for k in ("W_alpha", "H_alpha", "Z_alpha"):
            flat[f"{name}/{k}"] = np.array(float(fitkw.get(k, 1.0)))
        gi.pack(flat, name, "factors", **factor_args(V, W0, H0, scale=3, z=True))
        print(name, "n_iter", n_iter)
    # --- BetaMu over the convolutive modules (trainer.py:36-121 with NMFD / NMF2D / NMF3D as the single leaf) ---
    import torchnmf.trainer as ref_trainer
    for tag, cls, vshape, R, K in (("nmfd", "NMFD", (2, 21, 61), 5, (6,)), ("nmf2d", "NMF2D", (1, 3, 24, 31), 4, (4, 5)),
                                   ("nmf3d", "NMF3D", (1, 2, 10, 12, 14), 3, (2, 3, 4))):
        for beta in (0, 0.5, 1, 2):
            for reg, (l1, l2, ortho) in (("plain", (0, 0, 0)), ("reg", (0.1, 0.05, 0.2))):
                if reg == "reg" and beta not in (1, 2):
                    continue
                B, C, *X = vshape
                torch.manual_seed(0)
                V = torch.rand(*vshape).bfloat16().float() + (2 ** -7 if beta <= 0 else 0.0)
                torch.manual_seed(1)
                W0 = torch.randn(C, R, *K).abs(); H0 = torch.randn(B, R, *(x - k + 1 for x, k in zip(X, K))).abs()
                m = getattr(ref_nmf, cls)(W=W0, H=H0)
                tr = ref_trainer.BetaMu([m.W, m.H], beta, l1, l2, ortho)

                def closure():
                    tr.zero_grad()
                    return V, m()
                for _ in range(3):
                    tr.step(closure)
                name = f"betamu_{tag}_b{beta}_{reg}"
                for k, v in dict(V=V, W0=W0, H0=H0, W=m.W.detach().clone(), H=m.H.detach().clone(), gH=m.H.grad.clone()).items():
                    flat[f"{name}/{k}"] = v.numpy()
                for k, v in dict(beta=beta, l1=l1, l2=l2, ortho=ortho, steps=3, nd=len(K)).items():
                    flat[f"{name}/{k}"] = np.array(v, dtype=np.float64)
                gi.pack(flat, name, "factors", **factor_args(V, W0, H0, offset=2 ** -7 if beta <= 0 else 0.0))
    np.savez_compressed(os.path.join(GOLD, "reference_plca.npz"), **flat)
    print(f"wrote reference_plca.npz ({os.path.getsize(os.path.join(GOLD, 'reference_plca.npz')) / 1e6:.2f} MB)")


def sparse_cases():
    """Sparse-target NMF through the reference's own sparse path (nmf.py:603-638, :95-119), beta 1 and 2 (the branches that
    never form the dense product), target as in its tests/test_nmf_sparse.py:17-22 (entries above a threshold kept)."""
    torch.set_num_threads(1)
    cases = {}
    N, C, R = 300, 200, 8
    torch.manual_seed(0)
    D = torch.rand(N, C)
    D = torch.where(D > 0.93, D, torch.zeros(()))
    D[17] = 0                                   # an empty row and an empty column
    D[:, 5] = 0
    torch.manual_seed(1)
    W0, H0 = torch.randn(C, R).abs(), torch.randn(N, R).abs()
    Vs = D.to_sparse()
    for beta in (1, 2):
        for alpha, l1r in ((0, 0), (0.1, 0.5)):
            W, H, n_iter, losses = run_reference(ref_nmf.NMF, Vs, W0, H0, beta, float("-inf"), 20, alpha, l1r)
            cases[f"sparse_b{beta}_a{alpha}_l{l1r}"] = dict(
                kind="nmf", V=D, W0=W0, H0=H0, W=W, H=H, n_iter=n_iter, losses=losses,
                beta=beta, tol=float("-inf"), max_iter=20, alpha=alpha, l1_ratio=l1r)
        W, H, n_iter, losses = run_reference(ref_nmf.NMF, Vs, W0, H0, beta, 1e-3, 100, 0, 0)
        cases[f"sparse_b{beta}_stoprule"] = dict(kind="nmf", V=D, W0=W0, H0=H0, W=W, H=H, n_iter=n_iter, losses=losses,
                                                 beta=beta, tol=1e-3, max_iter=100, alpha=0, l1_ratio=0)
    save_cases(cases, "reference_sparse.npz", inputs=lambda c: (
        "thresholded", dict(shape=[N, C], rank=R, keep_above=0.93, seeds=[0, 1], empty_row=17, empty_col=5)))


def nd_cases():
    """NMF2D / NMF3D (nmf.py:782-942): ragged sizes, every beta branch, penalties, a batch of 2 and a frozen factor."""
    torch.set_num_threads(1)
    cases = {}
    specs = [("nmf2d", ref_nmf.NMF2D, (2, 5, 17, 23), 4, (3, 4)),
             ("nmf3d", ref_nmf.NMF3D, (1, 3, 9, 10, 21), 3, (2, 3, 5))]
    for kind, cls, vs, R, K in specs:
        B, C, X = vs[0], vs[1], vs[2:]
        hs = (B, R) + tuple(x - k + 1 for x, k in zip(X, K))
        for beta in (0, 0.5, 1, 1.5, 2, 3):
            for alpha, l1r in ((0, 0), (0.1, 0.5)):
                V, W0, H0 = make_inputs(vs, (C, R) + K, hs, floor=2 ** -7 if beta <= 0 else 0.0)
                W, H, n_iter, losses = run_reference(cls, V, W0, H0, beta, float("-inf"), 20, alpha, l1r)
                cases[f"{kind}_b{beta}_a{alpha}_l{l1r}"] = dict(
                    kind=kind, V=V, W0=W0, H0=H0, W=W, H=H, n_iter=n_iter, losses=losses,
                    beta=beta, tol=float("-inf"), max_iter=20, alpha=alpha, l1_ratio=l1r)
        V, W0, H0 = make_inputs(vs, (C, R) + K, hs)
        W, H, n_iter, losses = run_reference(cls, V, W0, H0, 1, 1e-3, 60, 0, 0)
        cases[f"{kind}_stoprule"] = dict(kind=kind, V=V, W0=W0, H0=H0, W=W, H=H, n_iter=n_iter, losses=losses,
                                         beta=1, tol=1e-3, max_iter=60, alpha=0, l1_ratio=0)
        W, H, n_iter, losses = run_reference(cls, V, W0, H0, 2, float("-inf"), 10, 0, 0, trainable_H=False)
        cases[f"{kind}_frozenH"] = dict(kind=kind, V=V, W0=W0, H0=H0, W=W, H=H, n_iter=n_iter, losses=losses,
                                        beta=2, tol=float("-inf"), max_iter=10, alpha=0, l1_ratio=0, trainable_H=False)
    # a kernel longer than one 32-wide shift chunk of the sliding axis, and outer axes longer than the kernel's
    vs, R, K = (1, 70, 6, 150), 5, (2, 37)
    V, W0, H0 = make_inputs(vs, (70, R) + K, (1, R, 5, 114))
    W, H, n_iter, losses = run_reference(ref_nmf.NMF2D, V, W0, H0, 1, float("-inf"), 10, 0, 0)
    cases["nmf2d_long_kernel"] = dict(kind="nmf2d", V=V, W0=W0, H0=H0, W=W, H=H, n_iter=n_iter, losses=losses,
                                      beta=1, tol=float("-inf"), max_iter=10, alpha=0, l1_ratio=0)
    save_cases(cases, "reference_nd.npz")


# Sparseness-constrained path (Hoyer 2004): _proj_func, sparse_fit, SparsityProj through the real reference
# ---------------------------------------------------------------------------------------------------------
def hoyer_cases():
    import torchnmf.trainer as ref_trainer
    from torchnmf.metrics import beta_div as ref_beta_div
    torch.set_num_threads(1)
    flat = {}

    def put(name, tensors, scalars):
        for k, v in tensors.items():
            flat[f"{name}/{k}"] = v.detach().numpy().copy()
        for k, v in scalars.items():
            flat[f"{name}/{k}"] = np.array(v, dtype=np.float64)

    # --- _proj_func on the slices of a parameter viewed as (outer, D, inner): unit-norm form and the line-search form ---
    for name, shape, dim, sp in (("proj_cols", (83, 8), 1, 0.5), ("proj_sparse", (257, 6), 1, 0.9),
                                 ("proj_slabs", (21, 4, 5), 1, 0.6), ("proj_dense", (64, 3), 1, 0.05),
                                 ("proj_big", (4099, 5), 1, 0.7), ("proj_dim0", (4, 300), 0, 0.8)):
        torch.manual_seed(3)
        X = torch.randn(*shape).abs() + 0.01
        if name == "proj_dim0":
            X[1] = torch.randn(300)                      # a slice with negative entries (a gradient step can produce them)
        D = shape[dim]
        n = X.numel() // D
        L1 = n ** 0.5 * (1 - sp) + sp
        norms = ref_nmf._get_norm(X, dim)
        for form, (k1, k2) in (("unit", ([L1] * D, [1.0] * D)),
                               ("scaled", ((L1 * norms).tolist(), (norms ** 2).tolist()))):
            Y = X.clone()
            for j in range(D):
                sl = (slice(None),) * dim + (j,)
                Y[sl] = ref_nmf._proj_func(X[sl].clone(), float(k1[j]), float(k2[j]))
            put(f"{name}_{form}", dict(X=X, Y=Y, k1=torch.tensor(k1, dtype=torch.float64),
                                       k2=torch.tensor(k2, dtype=torch.float64)), dict(dim=dim))
            gi.pack(flat, f"{name}_{form}", "proj_slices", shape=list(shape), negative_row=name == "proj_dim0")

    # --- sparse_fit (nmf.py:411-599) ---
    def run_sfit(name, cls, vshape, wshape, hshape, beta, iters, sW, sH, **kw):
        V, W0, H0 = make_inputs(vshape, wshape, hshape, floor=2 ** -7 if beta <= 0 else 0.0)
        m = cls(W=W0, H=H0, **kw)
        n_iter = m.sparse_fit(V, beta, iters, False, sW, sH)
        put(name, dict(V=V, W0=W0, H0=H0, W=m.W, H=m.H),
            dict(beta=beta, iters=iters, n_iter=n_iter, sW=-1 if sW is None else sW, sH=-1 if sH is None else sH,
                 trainable_W=int(kw.get("trainable_W", True)), trainable_H=int(kw.get("trainable_H", True))))
        gi.pack(flat, name, "factors", **factor_args(V, W0, H0, floor=2 ** -7 if beta <= 0 else 0.0))

    N, C, R = 97, 83, 8
    nmf = ref_nmf.NMF
    run_sfit("sfit_nmf_sW", nmf, (N, C), (C, R), (N, R), 2, 25, 0.5, None)
    run_sfit("sfit_nmf_sH", nmf, (N, C), (C, R), (N, R), 2, 25, None, 0.4)
    run_sfit("sfit_nmf_both", nmf, (N, C), (C, R), (N, R), 2, 25, 0.6, 0.3)
    run_sfit("sfit_nmf_kl_sW", nmf, (N, C), (C, R), (N, R), 1, 25, 0.3, None)      # (KL with both constraints ends in NaN in the reference)
    run_sfit("sfit_nmf_b15_both", nmf, (N, C), (C, R), (N, R), 1.5, 20, 0.5, 0.4)
    run_sfit("sfit_nmf_b05_sH", nmf, (N, C), (C, R), (N, R), 0.5, 20, None, 0.4)
    run_sfit("sfit_nmf_none", nmf, (N, C), (C, R), (N, R), 1, 20, None, None)
    run_sfit("sfit_nmf_frozenW", nmf, (N, C), (C, R), (N, R), 2, 20, 0.5, 0.4, trainable_W=False)
    run_sfit("sfit_nmf_frozenH", nmf, (N, C), (C, R), (N, R), 2, 20, 0.5, 0.4, trainable_H=False)
    run_sfit("sfit_nmf_mid", nmf, (1024, 512), (512, 32), (1024, 32), 2, 12, 0.5, 0.4)
    run_sfit("sfit_nmfd_sW", ref_nmf.NMFD, (2, 21, 61), (21, 4, 5), (2, 4, 57), 2, 20, 0.5, None)
    run_sfit("sfit_nmfd_kl_sH", ref_nmf.NMFD, (2, 21, 61), (21, 4, 5), (2, 4, 57), 1, 20, None, 0.4)
    run_sfit("sfit_nmf2d_both", ref_nmf.NMF2D, (1, 6, 20, 30), (6, 3, 3, 4), (1, 3, 18, 27), 2, 15, 0.5, 0.4)

    # --- sparse_fit on a SPARSE target (the reference's SDDMM derivation, nmf.py:603-638): this repo densifies such a target,
    # so the fixture pins "densified == the reference's sparse path" (its own tests/test_nmf_sparse.py:38-79 asserts the same
    # about itself).  Named spv_*: CPU tests only.
    for name, sW, sH in (("spv_sW", 0.3, None), ("spv_sH", None, 0.3)):
        torch.manual_seed(5)
        Vd = torch.rand(200, 150).bfloat16().float()
        Vd = Vd * (Vd > 0.9)
        torch.manual_seed(6)
        W0 = torch.randn(150, 8).abs(); H0 = torch.randn(200, 8).abs()
        m = ref_nmf.NMF(W=W0, H=H0)
        n_iter = m.sparse_fit(Vd.to_sparse(), 2, 8, False, sW, sH)
        put(name, dict(V=Vd, W0=W0, H0=H0, W=m.W, H=m.H),
            dict(beta=2, iters=8, n_iter=n_iter, sW=-1 if sW is None else sW, sH=-1 if sH is None else sH))
        gi.pack(flat, name, "thresholded", shape=[200, 150], rank=8, keep_above=0.9, seeds=[5, 6], bf16=True)

    # --- trainer.SparsityProj (trainer.py:124-190): steps on one NMF module, closure = beta_div of its reconstruction ---
    # (short runs: once the loss flattens, `loss <= init_loss` is decided by rounding and the step sizes of two
    # implementations part ways)
    # lr0 = 1 is the optimizer's default (the first steps walk through the halving branch); the others start from a step
    # size a user would set for this problem
    for name, which, beta, sp, steps, lr0 in (("sproj_W", "W", 2, 0.5, 4, 1.0), ("sproj_WH", "WH", 2, 0.4, 5, 1e-3),
                                              ("sproj_H", "H", 2, 0.6, 4, 1e-3)):
        V, W0, H0 = make_inputs((N, C), (C, R), (N, R))
        m = ref_nmf.NMF(W=W0, H=H0)
        params = [getattr(m, a) for a in which]
        tr = ref_trainer.SparsityProj(params, sp)
        tr.param_groups[0]["lr"] = lr0

        def closure():
            tr.zero_grad()
            return ref_beta_div(m(), V, beta)
        losses = [float(tr.step(closure)) for _ in range(steps)]
        put(name, dict(V=V, W0=W0, H0=H0, W=m.W, H=m.H, losses=torch.tensor(losses, dtype=torch.float64)),
            dict(beta=beta, sparsity=sp, steps=steps, lr0=lr0, lr=tr.param_groups[0]["lr"], on_W=int("W" in which), on_H=int("H" in which)))
        gi.pack(flat, name, "factors", **factor_args(V, W0, H0, floor=0.0))
    np.savez_compressed(os.path.join(GOLD, "reference_hoyer.npz"), **flat)
    print(f"wrote reference_hoyer.npz ({os.path.getsize(os.path.join(GOLD, 'reference_hoyer.npz')) / 1e6:.2f} MB)")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--cfg2", action="store_true")
    ap.add_argument("--only-cfg2", action="store_true")
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--r2", action="store_true", help="only the round-2 fixtures (reference_r2.npz)")
    ap.add_argument("--next-rows", action="store_true", help="only the BetaMu / PLCA fixtures (reference_next.npz)")
    ap.add_argument("--plca", action="store_true", help="only the SIPLCA / SIPLCA2 / SIPLCA3 fixtures (reference_plca.npz)")
    ap.add_argument("--sparse", action="store_true", help="only the sparse-target fixtures (reference_sparse.npz)")
    ap.add_argument("--hoyer", action="store_true", help="only the _proj_func / sparse_fit / SparsityProj fixtures (reference_hoyer.npz)")
    ap.add_argument("--nd", action="store_true", help="only the NMF2D / NMF3D fixtures (reference_nd.npz)")
    a = ap.parse_args()
    print("reference:", torchnmf.__file__, torchnmf.__version__, "torch", torch.__version__)
    if a.hoyer:
        hoyer_cases()
        sys.exit(0)
    if a.plca:
        plca_cases()
        sys.exit(0)
    if a.sparse:
        sparse_cases()
        sys.exit(0)
    if a.nd:
        nd_cases()
        sys.exit(0)
    if a.next_rows:
        next_row_cases()
        sys.exit(0)
    if a.r2:
        round2_cases()
        sys.exit(0)
    if not a.only_cfg2:
        save_cases(small_cases(), "reference_small.npz")
    if a.cfg2 or a.only_cfg2:
        cfg2_case(a.iters)
