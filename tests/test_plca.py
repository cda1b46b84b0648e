"""The PLCA family (SURVEY.md section 8 row f2): `plca.PLCA` and the shift-invariant `SIPLCA` / `SIPLCA2` / `SIPLCA3`
(reference: torchnmf/plca.py:193-625).

Fixtures: tests/golden/reference_next.npz (PLCA) and tests/golden/reference_plca.npz (SIPLCA*), written by
`python oracle/make_golden.py --next-rows / --plca` from the real torchnmf 0.3.5.

CPU tests: the closed-form oracle (oracle/plca_oracle.py) against those fixtures -- this is what pins it -- and the module
surface (constructors, shapes, normalisation, reconstruct).  GPU tests: `fit` through the C ABI
(`nmfb200_nmf_raw_terms` / `nmfb200_nmfd_raw_terms`) against the same fixtures at rtol 1e-3.
"""
import numpy as np
import pytest
import torch

from conftest import load_npz
from oracle import plca_oracle
from torchnmf_b200 import PLCA, SIPLCA, SIPLCA2, SIPLCA3, NMFD, NMF2D, NMF3D, BetaMu

ZN = load_npz("reference_next.npz")
ZP = load_npz("reference_plca.npz")
CLS = {0: PLCA, 1: SIPLCA, 2: SIPLCA2, 3: SIPLCA3}


def _case(name):
    z = ZN if name.startswith("plca_") else ZP
    c = {k.split("/", 1)[1]: z[k] for k in z.files if k.startswith(name + "/")}
    c.setdefault("cls", np.array(0)); c.setdefault("tol", np.array(float("-inf")))
    for k in ("trainable_W", "trainable_H"):
        c.setdefault(k, np.array(1))
    return c


def _t(c, k):
    return torch.from_numpy(c[k].copy())


NAMES = sorted({k.split("/")[0] for k in ZN.files if k.startswith("plca_")}
               | {k.split("/")[0] for k in ZP.files if k.startswith("siplca")})
BETAMU_ND = sorted({k.split("/")[0] for k in ZP.files if k.startswith("betamu_")})
SMALL = [n for n in NAMES if not n.endswith("_tc")]


def _close(got, want, rtol):
    return torch.allclose(got, want, rtol=rtol, atol=1e-5 * float(want.abs().max()))


def _worst(got, want):
    return float(((got - want).abs() / (want.abs() + 1e-5 * want.abs().max())).max())


# ---- CPU: the oracle is pinned by the reference's outputs ----------------------------------------------------------------
@pytest.mark.parametrize("name", SMALL)
def test_oracle_matches_reference(name):
    c = _case(name)
    mod = CLS[int(c["cls"])](W=_t(c, "W0"), H=_t(c, "H0"), Z=_t(c, "Z0"))        # the constructor normalises (plca.py:110-144)
    W, H, Z, n_iter, norm = plca_oracle.fit(
        _t(c, "V"), mod.W.data, mod.H.data, mod.Z.data, float(c["tol"]), int(c["iters"]),
        float(c["W_alpha"]), float(c["H_alpha"]), float(c["Z_alpha"]),
        bool(int(c["trainable_W"])), bool(int(c["trainable_H"])), bool(int(c["trainable_Z"])))
    assert n_iter == int(c["n_iter"]) and abs(float(norm) - float(c["norm"])) <= 1e-6 * float(c["norm"])
    for nm, got in (("W", W), ("H", H), ("Z", Z)):
        assert _close(got, _t(c, nm), 1e-4), (name, nm, _worst(got, _t(c, nm)))


def test_oracle_reconstruct_is_the_flipped_convolution():
    import torch.nn.functional as F
    torch.manual_seed(3)
    for cls, conv, vs, k in ((SIPLCA, F.conv1d, (2, 5, 19), (4,)), (SIPLCA2, F.conv2d, (1, 3, 9, 11), (2, 3)),
                             (SIPLCA3, F.conv3d, (1, 2, 6, 7, 8), (2, 3, 2))):
        m = cls(vs, 3, k if len(k) > 1 else k[0])
        ref = conv(m.H, m.W.flip(tuple(range(2, 2 + len(k)))) * m.Z.view(-1, *([1] * len(k))),
                   padding=tuple(x - 1 for x in k))                                   # plca.py:453-455, :534-537, :621-625
        assert torch.allclose(m(), ref, rtol=1e-5, atol=1e-8)
        assert torch.allclose(plca_oracle.reconstruct(m.H.data, m.W.data, m.Z.data), ref, rtol=1e-5, atol=1e-8)


# ---- CPU: module surface (the docstring examples of plca.py:413-425, :500-512, :584-596) ----------------------------------
def test_shift_invariant_module_surface():
    m = SIPLCA((1, 33, 50), 16, 3)
    assert m.W.shape == (33, 16, 3) and m.H.shape == (1, 16, 48) and m.Z.shape == (16,) and m().shape == (1, 33, 50)
    assert m.kernel_size == (3,) and m.out_channels == 33 and "kernel_size=(3,)" in repr(m)
    m = SIPLCA2((1, 1, 33, 50), 16, 3)
    assert m.W.shape == (1, 16, 3, 3) and m.H.shape == (1, 16, 31, 48) and m().shape == (1, 1, 33, 50)
    m = SIPLCA3((1, 3, 16, 16, 20), 8, (5, 5, 6))
    assert m.W.shape == (3, 8, 5, 5, 6) and m.H.shape == (1, 8, 12, 12, 15) and m().shape == (1, 3, 16, 16, 20)
    for mod in (SIPLCA((2, 7, 20), 4, 5), SIPLCA2((2, 3, 9, 10), 4, (2, 3))):
        dims = [d for d in range(mod.W.dim()) if d != 1]
        assert torch.allclose(mod.W.sum(dims), torch.ones(4), atol=1e-5)             # P(c, t | z) sums to one per component
        assert torch.allclose(mod.H.sum(dims), torch.ones(4), atol=1e-5)
        assert abs(float(mod().sum()) - 1) < 1e-4                                     # a joint distribution
    assert SIPLCA((1, 6, 9)).rank == 6 and SIPLCA((1, 6, 9)).W.shape == (6, 6, 1)     # rank = K, T = 1 defaults (plca.py:445-449)
    with pytest.raises(AssertionError, match="Latent size"):
        SIPLCA(W=torch.ones(4, 2, 3), H=torch.ones(1, 3, 5))
    with pytest.raises(AssertionError):
        SIPLCA(rank=None)
    with pytest.raises(ValueError):
        SIPLCA((33, 50), 16, 3)                                                       # wrong arity of Vshape


def _run_betamu(c, device, return_module):
    V = _t(c, "V").to(device)
    m = {1: NMFD, 2: NMF2D, 3: NMF3D}[int(c["nd"])](W=_t(c, "W0"), H=_t(c, "H0")).to(device)
    tr = BetaMu([m.W, m.H], float(c["beta"]), float(c["l1"]), float(c["l2"]), float(c["ortho"]))

    def closure():
        tr.zero_grad()
        return V, (m if return_module else m())
    paths = []
    for _ in range(int(c["steps"])):
        tr.step(closure)
        paths += tr.last_step_paths
    return m, paths


@pytest.mark.parametrize("name", BETAMU_ND)
def test_betamu_convolutive_autograd_path_matches_reference(name):
    c = _case(name)
    m, paths = _run_betamu(c, "cpu", False)
    assert set(paths) == {"autograd"}
    assert torch.allclose(m.W.data, _t(c, "W"), rtol=5e-5, atol=1e-7)
    assert torch.allclose(m.H.data, _t(c, "H"), rtol=5e-5, atol=1e-7)
    assert torch.allclose(m.H.grad, _t(c, "gH"), rtol=1e-4, atol=1e-5 * float(_t(c, "gH").abs().max()))


def test_fit_without_cuda_fails_loudly():
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        SIPLCA((1, 6, 9), 2, 3).fit(torch.rand(1, 6, 9))


# ---- GPU: fit through the C ABI ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", [n for n in NAMES if n.startswith("siplca")])
def test_siplca_fit_matches_reference(name):
    c = _case(name)
    m = CLS[int(c["cls"])](W=_t(c, "W0"), H=_t(c, "H0"), Z=_t(c, "Z0"), trainable_W=bool(int(c["trainable_W"])),
                           trainable_H=bool(int(c["trainable_H"])), trainable_Z=bool(int(c["trainable_Z"]))).cuda()
    n_iter, norm = m.fit(_t(c, "V").cuda(), float(c["tol"]), int(c["iters"]), False,
                         float(c["W_alpha"]), float(c["H_alpha"]), float(c["Z_alpha"]))
    assert m.last_fit_precision == "f32"
    assert n_iter == int(c["n_iter"]) and abs(float(norm) - float(c["norm"])) <= 1e-5 * float(c["norm"])
    for nm in ("W", "H", "Z"):
        got, want = getattr(m, nm).data.cpu(), _t(c, nm)
        assert _close(got, want, 1e-3), (name, nm, _worst(got, want))


@pytest.mark.gpu
@pytest.mark.parametrize("return_module", [False, True])
@pytest.mark.parametrize("name", BETAMU_ND)
def test_betamu_convolutive_fused_path_matches_reference(name, return_module):
    """BetaMu.step over an NMFD / NMF2D / NMF3D leaf takes both terms from nmfb200_nmfd_raw_terms (trainer.py:36-121)."""
    c = _case(name)
    m, paths = _run_betamu(c, "cuda", return_module)
    assert set(paths) == {"fused"}, paths
    for nm in ("W", "H"):
        got, want = getattr(m, nm).data.cpu(), _t(c, nm)
        assert _close(got, want, 1e-3), (name, nm, _worst(got, want))
    gH = _t(c, "gH")      # positive - negative term: judged against the terms' own magnitude (see tests/test_next_rows.py)
    assert torch.allclose(m.H.grad.cpu(), gH, rtol=2e-3, atol=1e-2 * float(gH.abs().max()))


@pytest.mark.gpu
def test_siplca_tensor_core_option():
    """precision="f16": the beta = 1 tcgen05 sliding GEMMs of NMFD under the EM step (opt-in, like PLCA's: the EM recursion
    keeps the fp16 operand rounding, so the bar here is 3e-3)."""
    c = _case("siplca_tc")
    m = SIPLCA(W=_t(c, "W0"), H=_t(c, "H0"), Z=_t(c, "Z0")).cuda()
    m.fit(_t(c, "V").cuda(), float("-inf"), int(c["iters"]), precision="f16")
    assert m.last_fit_precision == "f16"
    for nm in ("W", "H", "Z"):
        got, want = getattr(m, nm).data.cpu(), _t(c, nm)
        assert _close(got, want, 3e-3), (nm, _worst(got, want))


@pytest.mark.gpu
def test_siplca_host_module_and_double_are_staged():
    c = _case("siplca_small")
    m = SIPLCA(W=_t(c, "W0"), H=_t(c, "H0"), Z=_t(c, "Z0")).double()                # host-resident, float64
    m.fit(_t(c, "V").double(), float("-inf"), int(c["iters"]))
    assert m.W.dtype == torch.float64 and m.W.device.type == "cpu"
    for nm in ("W", "H", "Z"):
        assert _close(getattr(m, nm).data.float(), _t(c, nm), 1e-3)
