"""Pin the CPU oracle (oracle/mu_oracle.py) against outputs of the real reference.

The fixtures in tests/golden/reference_small.npz were produced by oracle/make_golden.py, which
imports torchnmf 0.3.5 from /root/reference and runs `fit` from identical initial factors.
"""
import math

import pytest
import torch

from conftest import load_golden
from oracle import mu_oracle as orc

CASES = load_golden()


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_matches_reference_fit(name):
    c = CASES[name]
    torch.set_num_threads(1)
    W, H, n_iter, losses = orc.fit(
        c["V"], c["W0"], c["H0"], beta=c["beta"], tol=c["tol"], max_iter=c["max_iter"],
        alpha=c["alpha"], l1_ratio=c["l1_ratio"],
        trainable_W=bool(c.get("trainable_W", 1)), trainable_H=bool(c.get("trainable_H", 1)),
        kind=c["kind"])
    assert n_iter == c["n_iter"]
    # closed form vs autograd: identical maths, reduction order differs only inside BLAS calls.
    # beta outside [1, 2] takes a gamma-th root (pow), the loosest branch.
    rtol = 2e-5 if c["kind"] == "nmf" else 5e-5
    assert torch.allclose(W, c["W"], rtol=rtol, atol=1e-7), (W - c["W"]).abs().max()
    assert torch.allclose(H, c["H"], rtol=rtol, atol=1e-7), (H - c["H"]).abs().max()
    assert len(losses) == len(c["losses"])
    for a, b in zip(losses, c["losses"]):
        assert math.isclose(a, b, rel_tol=1e-4, abs_tol=1e-6)


def test_frozen_factor_is_untouched():
    c = CASES["nmf_frozenW"]
    assert torch.equal(c["W"], c["W0"])          # the reference itself left W alone
    W, H, _, _ = orc.fit(c["V"], c["W0"], c["H0"], beta=c["beta"], tol=c["tol"], max_iter=c["max_iter"],
                         trainable_W=False)
    assert torch.equal(W, c["W0"])


@pytest.mark.parametrize("beta", [-1, 0, 0.5, 1, 1.5, 2, 3])
def test_beta_div_nonneg_and_zero_at_equality(beta):
    # tests/test_metrics.py:6-14 of the reference: beta_div >= 0, no NaN
    torch.manual_seed(0)
    x = torch.rand(50, 40) + 0.1
    y = torch.rand(50, 40) + 0.1
    d = orc.beta_div(x, y, beta)
    assert not torch.isnan(d) and d >= -1e-4
    assert abs(float(orc.beta_div(y, y, beta))) < 1e-2


def test_beta_le0_with_zeros_raises():
    V = torch.rand(10, 10)
    V[0, 0] = 0
    with pytest.raises(ValueError):
        orc.fit(V, torch.rand(10, 3), torch.rand(10, 3), beta=0)


def test_nmfd_reconstruct_matches_definition():
    # nmf.py:712-713: V[i,j] ~= sum_t sum_r W[i,r,t] H[r,j-t]
    torch.manual_seed(0)
    W = torch.rand(5, 3, 4)
    H = torch.rand(2, 3, 7)
    out = orc.nmfd_reconstruct(H, W)
    ref = torch.zeros(2, 5, 10)
    for b in range(2):
        for i in range(5):
            for j in range(10):
                for t in range(4):
                    if 0 <= j - t < 7:
                        ref[b, i, j] += (W[i, :, t] * H[b, :, j - t]).sum()
    assert torch.allclose(out, ref, atol=1e-5)


def test_sharded_w_contractions_sum_to_full():
    # SURVEY 8e: row shards of (V, H) give partial numerators that add up (before relu/eps/l1/l2).
    torch.manual_seed(0)
    V = torch.rand(64, 30); W = torch.rand(30, 5); H = torch.rand(64, 5)
    for beta in (0.5, 1, 2):
        num, den = orc.nmf_w_contractions(V, W, H, beta)
        n0, d0 = orc.nmf_w_contractions(V[:40], W, H[:40], beta)
        n1, d1 = orc.nmf_w_contractions(V[40:], W, H[40:], beta)
        assert torch.allclose(n0 + n1, num, rtol=1e-5, atol=1e-6)
        assert torch.allclose(d0 + d1, den, rtol=1e-5, atol=1e-6)


# ---- round-2 fixtures (tests/golden/reference_r2.npz): the oracle at the config shapes --------------------------
import os  # noqa: E402

import numpy as np  # noqa: E402

from conftest import GOLDEN  # noqa: E402

_Z2 = np.load(os.path.join(GOLDEN, "reference_r2.npz"), allow_pickle=False)


def _r2_case(name):
    return {k.split("/", 1)[1]: _Z2[k] for k in _Z2.files if k.startswith(name + "/")}


def _r2_inputs(shape_v, shape_w, shape_h, floor=0.0):
    torch.manual_seed(0)
    V = torch.rand(*shape_v).bfloat16().float()
    if floor > 0:
        V = V.clamp_min(floor)
    torch.manual_seed(1)
    return V, torch.randn(*shape_w).abs(), torch.randn(*shape_h).abs()


@pytest.mark.parametrize("name", ["nmfd_ragged_b1", "nmfd_ragged_b0.5", "nmf_sweep_b0", "nmf_sweep_b0.5",
                                  "nmf_sweep_b1.5", "nmf_sweep_b2"])
def test_oracle_matches_reference_round2_fixtures(name):
    c = _r2_case(name)
    torch.set_num_threads(os.cpu_count())
    if name.startswith("nmfd"):
        B, C, L, R, T = (int(c[k]) for k in ("B", "C", "L", "R", "T"))
        V, W0, H0 = _r2_inputs((B, C, L), (C, R, T), (B, R, L - T + 1))
        kind = "nmfd"
    else:
        N, C, R = int(c["N"]), int(c["C"]), int(c["R"])
        V, W0, H0 = _r2_inputs((N, C), (C, R), (N, R), floor=float(c["floor"]))
        kind = "nmf"
    assert math.isclose(V.double().sum().item(), float(c["v_sum"]), rel_tol=1e-12)
    W, H, n_iter, losses = orc.fit(V, W0, H0, beta=float(c["beta"]), tol=float("-inf"), max_iter=int(c["max_iter"]),
                                   kind=kind)
    assert n_iter == int(c["n_iter"])
    ws, hs = int(c["w_step"]), int(c["h_step"])
    Hs = H[::hs] if H.dim() == 2 else H[..., ::hs]
    # 50 iterations, multi-threaded BLAS on both sides: reduction order differs -> 2e-4
    assert torch.allclose(W[::ws], torch.from_numpy(c["W_sub"]), rtol=2e-4, atol=1e-6 * float(c["w_absmax"]))
    assert torch.allclose(Hs, torch.from_numpy(c["H_sub"]), rtol=2e-4, atol=1e-6 * float(c["h_absmax"]))


ND_CASES = load_golden("reference_nd.npz")


@pytest.mark.parametrize("name", sorted(ND_CASES))
def test_oracle_matches_reference_nmf2d_nmf3d(name):
    """NMF2D / NMF3D (nmf.py:782-942): the shifted-product restatement against fits of the real reference."""
    c = ND_CASES[name]
    torch.set_num_threads(1)
    W, H, n_iter, losses = orc.fit(
        c["V"], c["W0"], c["H0"], beta=c["beta"], tol=c["tol"], max_iter=c["max_iter"],
        alpha=c["alpha"], l1_ratio=c["l1_ratio"],
        trainable_W=bool(c.get("trainable_W", 1)), trainable_H=bool(c.get("trainable_H", 1)), kind=c["kind"])
    assert n_iter == c["n_iter"]
    assert torch.allclose(W, c["W"], rtol=1e-4, atol=1e-7), (W - c["W"]).abs().max()
    assert torch.allclose(H, c["H"], rtol=1e-4, atol=1e-7), (H - c["H"]).abs().max()
    assert len(losses) == len(c["losses"])
    for a, b in zip(losses, c["losses"]):
        assert math.isclose(a, b, rel_tol=1e-4, abs_tol=1e-6)


def test_nmfnd_reconstruct_is_the_full_convolution():
    """The shifted-product form equals conv2d / conv3d with the flipped kernel and full padding (nmf.py:861-865, :938-942)."""
    import torch.nn.functional as F
    torch.manual_seed(0)
    H, W = torch.rand(2, 3, 6, 7), torch.rand(4, 3, 2, 3)
    assert torch.allclose(orc.nmfnd_reconstruct(H, W), F.conv2d(H, W.flip((2, 3)), padding=(1, 2)), atol=1e-5)
    H, W = torch.rand(1, 2, 4, 5, 6), torch.rand(3, 2, 2, 2, 3)
    assert torch.allclose(orc.nmfnd_reconstruct(H, W), F.conv3d(H, W.flip((2, 3, 4)), padding=(1, 1, 2)), atol=1e-5)


SP_CASES = load_golden("reference_sparse.npz")


@pytest.mark.parametrize("name", sorted(SP_CASES))
def test_oracle_on_the_dense_target_matches_reference_sparse_fit(name):
    """The reference's sparse path (nmf.py:603-638, :95-119) is the dense update on V.to_dense() (its own
    tests/test_nmf_sparse.py:8-37): the dense oracle reproduces fits the reference ran on the SPARSE target."""
    c = SP_CASES[name]
    torch.set_num_threads(1)
    W, H, n_iter, losses = orc.fit(c["V"], c["W0"], c["H0"], beta=c["beta"], tol=c["tol"], max_iter=c["max_iter"],
                                   alpha=c["alpha"], l1_ratio=c["l1_ratio"])
    assert n_iter == c["n_iter"]
    assert torch.allclose(W, c["W"], rtol=1e-4, atol=1e-7), (W - c["W"]).abs().max()
    assert torch.allclose(H, c["H"], rtol=1e-4, atol=1e-7), (H - c["H"]).abs().max()
    for a, b in zip(losses, c["losses"]):
        assert math.isclose(a, b, rel_tol=1e-4, abs_tol=1e-5)
