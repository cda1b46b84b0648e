"""GPU parity at the shapes of BASELINE.json configs[2..4] against reference-generated goldens
(tests/golden/reference_r2.npz, written by `python oracle/make_golden.py --r2` from the real torchnmf 0.3.5).

Inputs are regenerated from the fixture's seeds and verified against its float64 checksums; only subsampled
factors are stored (rows at a stride, the H of NMFD along its last axis).  Tolerance everywhere: the north-star's
rtol 1e-3 with atol = 1e-5 * max|factor| for the near-zero entries multiplicative updates produce.
"""
import math
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from torchnmf_b200 import NMF, NMFD

pytestmark = pytest.mark.gpu
RTOL, ATOL_REL = 1e-3, 1e-5
Z = np.load(os.path.join(GOLDEN, "reference_r2.npz"), allow_pickle=False)


def _case(name):
    return {k.split("/", 1)[1]: Z[k] for k in Z.files if k.startswith(name + "/")}


def _inputs(shape_v, shape_w, shape_h, floor=0.0, heavy=False):
    torch.manual_seed(0)
    if heavy:
        V = torch.exp(2.0 * torch.randn(*shape_v)).bfloat16().float()
    else:
        V = torch.rand(*shape_v).bfloat16().float()
    if floor > 0:
        V = V.clamp_min(floor)
    torch.manual_seed(1)
    W0 = torch.randn(*shape_w).abs()
    H0 = torch.randn(*shape_h).abs()
    return V, W0, H0


def _check_inputs(c, V, W0, H0):
    assert math.isclose(V.double().sum().item(), float(c["v_sum"]), rel_tol=1e-12)
    assert math.isclose(W0.double().sum().item(), float(c["w0_sum"]), rel_tol=1e-12)
    assert math.isclose(H0.double().sum().item(), float(c["h0_sum"]), rel_tol=1e-12)


def _compare(c, m, label, rtol=RTOL):
    ws, hs = int(c["w_step"]), int(c["h_step"])
    W = m.W.data.cpu()[::ws]
    H = m.H.data.cpu()
    H = H[::hs] if H.dim() == 2 else H[..., ::hs]
    worst = 0.0
    for got, want, mx, nm in ((W, torch.from_numpy(c["W_sub"]), float(c["w_absmax"]), "W"),
                              (H, torch.from_numpy(c["H_sub"]), float(c["h_absmax"]), "H")):
        atol = ATOL_REL * mx
        err = ((got - want).abs() / (rtol * want.abs() + atol)).max().item()
        worst = max(worst, err)
        assert err <= 1.0, f"{label} {nm}: {err:.2f} x tolerance (rtol {rtol}, atol {atol:.2e})"
    return worst


@pytest.mark.parametrize("name", ["nmfd_cfg3", "nmfd_ragged_b1", "nmfd_ragged_b0.5"])
@pytest.mark.parametrize("precision", ["auto", "f32"])
def test_nmfd_matches_reference_at_config_shapes(name, precision):
    """cfg3 (1025 x 8192, R = 16, T = 128: four 32-wide shift chunks, nine 128-row tiles) and a ragged case
    (T = 37, C = 130, batch 2).  Reference: nmf.py:776-779 + the fit loop."""
    c = _case(name)
    B, C, L, R, T = (int(c[k]) for k in ("B", "C", "L", "R", "T"))
    V, W0, H0 = _inputs((B, C, L), (C, R, T), (B, R, L - T + 1))
    _check_inputs(c, V, W0, H0)
    m = NMFD(W=W0, H=H0).cuda()
    n = m.fit(V.cuda(), float(c["beta"]), float("-inf"), int(c["max_iter"]), precision=precision)
    assert n == int(c["n_iter"])
    _compare(c, m, f"{name} [{m.last_fit_precision}]")


@pytest.mark.parametrize("precision", ["auto", "f16_split", "f32"])
def test_rank128_kl_100_iterations_match_reference(precision):
    """The R = 128 operand kernels (cfg4's per-GPU kernel) over 100 KL iterations at 8192 x 2048."""
    c = _case("nmf_r128_kl")
    N, C, R = int(c["N"]), int(c["C"]), int(c["R"])
    V, W0, H0 = _inputs((N, C), (C, R), (N, R))
    _check_inputs(c, V, W0, H0)
    m = NMF(W=W0, H=H0).cuda()
    n = m.fit(V.cuda(), 1, float("-inf"), int(c["max_iter"]), precision=precision)
    assert n == int(c["n_iter"])
    if precision != "f32":
        assert m.last_fit_precision == ("f16" if precision == "auto" else precision)
    _compare(c, m, f"r128 [{m.last_fit_precision}]")


@pytest.mark.parametrize("beta", [0, 0.5, 1.5, 2])
@pytest.mark.parametrize("precision", ["auto", "f16_split", "f32"])
def test_beta_sweep_50_iterations_match_reference(beta, precision):
    """cfg5-shaped sweep (4096 x 1024, R = 64, 50 iterations) for every beta branch of nmf.py:61-74, default precision
    included, at the north-star tolerance."""
    c = _case(f"nmf_sweep_b{beta}")
    N, C, R = int(c["N"]), int(c["C"]), int(c["R"])
    V, W0, H0 = _inputs((N, C), (C, R), (N, R), floor=float(c["floor"]))
    _check_inputs(c, V, W0, H0)
    m = NMF(W=W0, H=H0).cuda()
    n = m.fit(V.cuda(), beta, float("-inf"), int(c["max_iter"]), precision=precision)
    assert n == int(c["n_iter"])
    _compare(c, m, f"sweep beta={beta} [{m.last_fit_precision}]")


@pytest.mark.parametrize("beta", [1, 0])
def test_heavy_tailed_target_default_precision_matches_reference(beta):
    """Lognormal target spanning ~6 decades (spectrogram-like): `auto` must not silently lose the small entries to
    the fp16 operand range -- whatever arithmetic it resolves to has to hold the parity bar."""
    c = _case(f"nmf_heavy_b{beta}")
    N, C, R = int(c["N"]), int(c["C"]), int(c["R"])
    V, W0, H0 = _inputs((N, C), (C, R), (N, R), heavy=True)
    _check_inputs(c, V, W0, H0)
    m = NMF(W=W0, H=H0).cuda()
    n = m.fit(V.cuda(), beta, float("-inf"), int(c["max_iter"]))
    assert n == int(c["n_iter"])
    _compare(c, m, f"heavy beta={beta} [{m.last_fit_precision}]")


def test_nmfd_tensor_core_fit_is_bitwise_repeatable():
    """Two fits from the same state give identical bits: every reduction of the tensor-core NMFD path runs in a fixed
    order (split partials summed in order, the only atomics are integer max), and the shared-memory windows are handed
    over by mbarriers -- a lost ordering there would show up here as run-to-run differences."""
    torch.manual_seed(3)
    V = torch.rand(2, 130, 700).cuda()
    W0 = torch.rand(130, 5, 37)
    H0 = torch.rand(2, 5, 700 - 37 + 1)
    outs = []
    for _ in range(3):
        m = NMFD(W=W0.clone(), H=H0.clone()).cuda()
        m.fit(V, 1, float("-inf"), 12)
        assert m.last_fit_precision == "f16"
        outs.append((m.W.data.clone(), m.H.data.clone()))
    for W, H in outs[1:]:
        assert torch.equal(W, outs[0][0]) and torch.equal(H, outs[0][1])


# ---- the loss folded into the W update's contraction pass (nmfb200_nmf_loss_prefetch_w) -----------------------------------
def _kl_engine(N, C, R):
    from torchnmf_b200 import engine as _engine
    V, W0, H0 = _inputs((N, C), (C, R), (N, R))
    W, H = W0.cuda(), H0.cuda()
    return _engine.CudaNmfEngine(V.cuda(), W, H, "f16"), W, H


@pytest.mark.parametrize("shape", [(1000, 777, 64), (640, 512, 128), (300, 260, 40)])
def test_prefetched_loss_equals_the_loss_pass_and_feeds_the_next_w_update(shape):
    """The fold computes the LOSS kernel's sums from the W contraction's own S tiles: same value (summation order aside), and
    the W update that follows, which skips its contraction, gives the bits of a plain W update."""
    N, C, R = shape
    eng, W, H = _kl_engine(N, C, R)
    try:
        for _ in range(3):
            eng.update_w(1.0, 1.0, 0.0, 0.0)
            eng.update_h(1.0, 1.0, 0.0, 0.0)
        want = eng.loss(1.0)
        W_before = W.clone()
        eng.update_w(1.0, 1.0, 0.0, 0.0)
        W_plain = W.clone()
        W.copy_(W_before)
        eng.sync()
        got = eng.loss_prefetch_w(1.0)
        assert got == pytest.approx(want, rel=2e-6)
        eng.update_w(1.0, 1.0, 0.0, 0.0)                    # reuses the prefetched numerators
        assert torch.equal(W, W_plain)
        # a prefetch that is NOT followed by the W update is dropped: H update, then a fresh W update
        W.copy_(W_before)
        eng.sync()
        eng.update_h(1.0, 1.0, 0.0, 0.0)
        eng.update_w(1.0, 1.0, 0.0, 0.0)
        W_seq = W.clone()
        H_seq = H.clone()
    finally:
        eng.close()
    eng2, W2, H2 = _kl_engine(N, C, R)
    try:
        for _ in range(3):
            eng2.update_w(1.0, 1.0, 0.0, 0.0)
            eng2.update_h(1.0, 1.0, 0.0, 0.0)
        eng2.loss_prefetch_w(1.0)
        eng2.update_h(1.0, 1.0, 0.0, 0.0)                   # overwrites the partial numerators: the prefetch must not be used
        eng2.update_w(1.0, 1.0, 0.0, 0.0)
    finally:
        eng2.close()
    # eng ran one extra H update before this point (the one inside the loop body above is shared): compare like with like
    eng3, W3, H3 = _kl_engine(N, C, R)
    try:
        for _ in range(3):
            eng3.update_w(1.0, 1.0, 0.0, 0.0)
            eng3.update_h(1.0, 1.0, 0.0, 0.0)
        eng3.update_h(1.0, 1.0, 0.0, 0.0)
        eng3.update_w(1.0, 1.0, 0.0, 0.0)
    finally:
        eng3.close()
    assert torch.equal(W2, W3) and torch.equal(H2, H3)
    assert torch.equal(W_seq, W3) and torch.equal(H_seq, H3)


def test_fit_with_the_folded_loss_is_the_fit_with_the_loss_pass(monkeypatch):
    """Same factors, same losses, same stop decisions whether every 10th iteration's loss comes out of the next W update's
    contraction or out of a pass of its own; a stop right after a prefetch leaves the factors of that iteration."""
    from torchnmf_b200 import engine as _engine
    V, W0, H0 = _inputs((2048, 1024), (1024, 64), (2048, 64))
    a = NMF(W=W0, H=H0).cuda()
    na = a.fit(V.cuda(), 1, float("-inf"), 35, precision="f16")
    monkeypatch.delattr(_engine.CudaNmfEngine, "loss_prefetch_w")
    b = NMF(W=W0, H=H0).cuda()
    nb = b.fit(V.cuda(), 1, float("-inf"), 35, precision="f16")
    monkeypatch.undo()
    assert na == nb == 35
    assert torch.equal(a.W.data, b.W.data) and torch.equal(a.H.data, b.H.data)
    c = NMF(W=W0, H=H0).cuda()
    nc = c.fit(V.cuda(), 1, 1e9, 35, precision="f16")          # the stop rule fires at the first evaluation (iteration 10)
    d = NMF(W=W0, H=H0).cuda()
    nd = d.fit(V.cuda(), 1, float("-inf"), 10, precision="f16")
    assert nc == nd == 10
    assert torch.equal(c.W.data, d.W.data) and torch.equal(c.H.data, d.H.data)
