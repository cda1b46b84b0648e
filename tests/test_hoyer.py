"""Sparseness-constrained path (Hoyer 2004): `_proj_func` (nmf.py:21-49), `BaseComponent.sparse_fit` (nmf.py:411-599),
`trainer.SparsityProj` (trainer.py:124-190), `metrics.sparseness`, `utils`.  Fixtures: tests/golden/reference_hoyer.npz,
written by `python oracle/make_golden.py --hoyer` from the real torchnmf 0.3.5.

CPU tests: the oracle restatement (oracle/hoyer_oracle.py) against the reference's outputs; the host logic of `sparse_fit`
and `SparsityProj` with the oracle standing in for the library.  GPU tests: `nmfb200_hoyer_project`, `sparse_fit` and
`SparsityProj` through the C ABI against the same fixtures (rtol 1e-3, atol 1e-5 * max: the north-star tolerance).
"""
import numpy as np
import pytest
import torch

from conftest import load_npz
from oracle import hoyer_oracle as hoy
from oracle import mu_oracle as orc
from oracle_engine import OracleNmfEngine, OracleNmfdEngine
import torchnmf_b200
from torchnmf_b200 import NMF, NMF2D, NMFD, SparsityProj
from torchnmf_b200 import engine as _engine
from torchnmf_b200 import trainer as _trainer
from torchnmf_b200.metrics import beta_div, sparseness

Z = load_npz("reference_hoyer.npz")
NAMES = sorted({k.split("/")[0] for k in Z.files})
PROJ = [n for n in NAMES if n.startswith("proj_")]
SFIT = [n for n in NAMES if n.startswith("sfit_")]
SPROJ = [n for n in NAMES if n.startswith("sproj_")]
CLS = {"nmf": NMF, "nmfd": NMFD, "nmf2d": NMF2D}


def _case(name):
    return {k.split("/", 1)[1]: Z[k] for k in Z.files if k.startswith(name + "/")}


def _t(c, k):
    return torch.from_numpy(c[k].copy())


def _kind(name):
    return name.split("_")[1]


def _opt(c, k):
    return None if float(c[k]) < 0 else float(c[k])


# Entries next to the projection's zeroing threshold amplify rounding: on this case the restatement itself sits 7e-5 * max
# from the reference (every other case: <= 5e-6), so it is held to the north-star tolerance instead of the oracle's.
LOOSE = {"sfit_nmf_both": (1e-3, 1e-5)}
ORACLE_TOL = (2e-4, 1e-5)      # rtol, atol / max|x| (entries the projection leaves next to zero carry absolute, not relative, error)


def _err(got, want, rtol, atol_rel):
    atol = atol_rel * float(want.abs().max())
    return ((got - want).abs() / (rtol * want.abs() + atol)).max().item()


# ------------------------------------------------------------------------------------------------------------------
# CPU: the oracle is pinned to the reference
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", PROJ)
def test_oracle_projection_matches_reference(name):
    c = _case(name)
    Y = hoy.project_slices(_t(c, "X"), int(c["dim"]), c["k1"], c["k2"])
    assert _err(Y, _t(c, "Y"), 1e-5, 5e-6) <= 1.0


@pytest.mark.parametrize("name", SFIT)
def test_oracle_sparse_fit_matches_reference(name):
    c = _case(name)
    kind = {"nmf": "nmf", "nmfd": "nmfd", "nmf2d": "nmfnd"}[_kind(name)]
    W, H, n_iter, _ = hoy.sparse_fit(_t(c, "V"), _t(c, "W0"), _t(c, "H0"), float(c["beta"]), int(c["iters"]), _opt(c, "sW"),
                                    _opt(c, "sH"), bool(c["trainable_W"]), bool(c["trainable_H"]), kind)
    assert n_iter == int(c["n_iter"])
    tol = LOOSE.get(name, ORACLE_TOL)
    assert _err(W, _t(c, "W"), *tol) <= 1.0
    assert _err(H, _t(c, "H"), *tol) <= 1.0


def _oracle_sproj(c):
    V, W, H = _t(c, "V"), _t(c, "W0").clone(), _t(c, "H0").clone()
    beta, lr = float(c["beta"]), float(c["lr0"])
    losses = []
    for _ in range(int(c["steps"])):
        G = hoy.dloss_dwh(V, orc.nmf_reconstruct(H, W), beta)
        params, grads = [], []
        if int(c["on_W"]):
            params.append(W); grads.append(G.t() @ H)
        if int(c["on_H"]):
            params.append(H); grads.append(G @ W)
        loss, lr = hoy.sparsity_proj_step(params, grads, lambda: orc.beta_div(orc.nmf_reconstruct(H, W), V, beta),
                                          float(c["sparsity"]), lr)
        losses.append(float(loss))
    return W, H, lr, losses


@pytest.mark.parametrize("name", SPROJ)
def test_oracle_sparsity_proj_matches_reference(name):
    c = _case(name)
    W, H, lr, losses = _oracle_sproj(c)
    assert lr == pytest.approx(float(c["lr"]), rel=1e-12)
    assert np.allclose(losses, c["losses"], rtol=1e-5)
    assert _err(W, _t(c, "W"), *ORACLE_TOL) <= 1.0 and _err(H, _t(c, "H"), *ORACLE_TOL) <= 1.0


# ------------------------------------------------------------------------------------------------------------------
# CPU: host logic of sparse_fit / SparsityProj with the oracle in place of the library
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", [n for n in SFIT if _kind(n) in ("nmf", "nmfd") and n != "sfit_nmf_mid"])
def test_sparse_fit_host_logic_matches_reference(name):
    c = _case(name)
    m = CLS[_kind(name)](W=_t(c, "W0"), H=_t(c, "H0"), trainable_W=bool(c["trainable_W"]), trainable_H=bool(c["trainable_H"]))
    m._engine_factory = OracleNmfEngine if _kind(name) == "nmf" else OracleNmfdEngine
    n_iter = m.sparse_fit(_t(c, "V"), float(c["beta"]), int(c["iters"]), False, _opt(c, "sW"), _opt(c, "sH"))
    assert n_iter == int(c["n_iter"])
    tol = LOOSE.get(name, ORACLE_TOL)
    assert _err(m.W.data, _t(c, "W"), *tol) <= 1.0
    assert _err(m.H.data, _t(c, "H"), *tol) <= 1.0


@pytest.mark.parametrize("name", [n for n in NAMES if n.startswith("spv_")])
def test_sparse_fit_on_a_sparse_target_is_the_references_sparse_path(name):
    """The reference ran these through its sparse (SDDMM) derivation, nmf.py:603-638; here a sparse target of `sparse_fit` is
    densified: the oracle on the dense matrix and the host logic on the COO tensor both land on the reference's factors."""
    c = _case(name)
    V = _t(c, "V")
    W, H, n_iter, _ = hoy.sparse_fit(V, _t(c, "W0"), _t(c, "H0"), 2, int(c["iters"]), _opt(c, "sW"), _opt(c, "sH"))
    assert n_iter == int(c["n_iter"])
    assert _err(W, _t(c, "W"), *ORACLE_TOL) <= 1.0 and _err(H, _t(c, "H"), *ORACLE_TOL) <= 1.0
    m = NMF(W=_t(c, "W0"), H=_t(c, "H0"))
    m._engine_factory = OracleNmfEngine
    m.sparse_fit(V.to_sparse(), 2, int(c["iters"]), False, _opt(c, "sW"), _opt(c, "sH"))
    assert _err(m.W.data, _t(c, "W"), *ORACLE_TOL) <= 1.0 and _err(m.H.data, _t(c, "H"), *ORACLE_TOL) <= 1.0


@pytest.mark.parametrize("name", SPROJ)
def test_sparsity_proj_host_logic_matches_reference(name, monkeypatch):
    c = _case(name)
    monkeypatch.setattr(_trainer, "_project_slices_",
                        lambda p, dim, k1, k2: p.copy_(hoy.project_slices(p, dim, k1, k2)))
    V = _t(c, "V")
    m = NMF(W=_t(c, "W0"), H=_t(c, "H0"))
    tr = SparsityProj([p for p, on in ((m.W, c["on_W"]), (m.H, c["on_H"])) if int(on)], float(c["sparsity"]))
    tr.param_groups[0]["lr"] = float(c["lr0"])

    def closure():
        tr.zero_grad()
        return beta_div(m(), V, float(c["beta"]))
    losses = [float(tr.step(closure)) for _ in range(int(c["steps"]))]
    assert tr.param_groups[0]["lr"] == pytest.approx(float(c["lr"]), rel=1e-12)
    assert np.allclose(losses, c["losses"], rtol=1e-5)
    assert _err(m.W.data, _t(c, "W"), *ORACLE_TOL) <= 1.0 and _err(m.H.data, _t(c, "H"), *ORACLE_TOL) <= 1.0


def test_surface_and_errors():
    import inspect
    sig = inspect.signature(NMF.sparse_fit)
    assert list(sig.parameters)[:7] == ["self", "V", "beta", "max_iter", "verbose", "sW", "sH"]      # nmf.py:412-419
    assert sig.parameters["beta"].default == 2 and sig.parameters["max_iter"].default == 200
    with pytest.raises(ValueError, match="Invalid sparsity"):
        SparsityProj([torch.nn.Parameter(torch.rand(3, 2))], 1.0)
    with pytest.raises(ValueError, match="Invalid sparsity"):
        SparsityProj([torch.nn.Parameter(torch.rand(3, 2))], 0.0)
    opt = SparsityProj([torch.nn.Parameter(torch.rand(3, 2))], 0.5)
    assert opt.defaults == dict(sparsity=0.5, lr=1, dim=1, max_iter=10)                              # trainer.py:143-147
    m = NMF(W=torch.rand(5, 2), H=torch.rand(4, 2))
    m._engine_factory = OracleNmfEngine
    V = torch.rand(4, 5)
    V[0, 0] = 0
    with pytest.raises(ValueError, match="beta <= 0"):
        m.sparse_fit(V, beta=0, max_iter=1)
    with pytest.raises(AssertionError, match="non-negative"):
        m.sparse_fit(-V, beta=2, max_iter=1)
    with pytest.raises(TypeError):                      # the library projects CUDA tensors only: no CPU path
        _engine.hoyer_project_(torch.rand(4, 2), 1, [1.0, 1.0], [1.0, 1.0])
    x = torch.rand(7, 3)
    assert torch.allclose(torchnmf_b200.utils.normalize(x, 0).sum(0), torch.ones(3))
    y = x.clone()
    torchnmf_b200.utils.renorm_(y, 1)
    assert torch.allclose(y, x / (x * x).sum(0, keepdim=True))
    assert float(sparseness(torch.tensor([0., 0., 3., 0.]))) == pytest.approx(1.0)
    assert float(sparseness(torch.ones(9))) == pytest.approx(0.0, abs=1e-6)


def test_projected_slices_have_the_requested_sparseness():
    c = _case("proj_cols_unit")
    Y = _t(c, "Y")
    n = Y.shape[0]
    want = (n ** 0.5 - float(c["k1"][0])) / (n ** 0.5 - 1)        # k1 = sqrt(n) (1 - s) + s, unit L2 norm
    for j in range(Y.shape[1]):
        assert float(sparseness(Y[:, j])) == pytest.approx(want, abs=1e-5)
        assert float(Y[:, j].min()) >= 0


# ------------------------------------------------------------------------------------------------------------------
# GPU: through the C ABI
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", PROJ)
def test_projection_kernel_matches_reference(name):
    c = _case(name)
    x = _t(c, "X").cuda()
    _engine.hoyer_project_(x, int(c["dim"]), c["k1"], c["k2"])
    torch.cuda.synchronize()
    assert _err(x.cpu(), _t(c, "Y"), 1e-4, 5e-6) <= 1.0


@pytest.mark.gpu
def test_projection_kernel_large_slices_match_oracle():
    """65536-element strided slices (the H of BASELINE configs[1]), several rounds of zeroing; three slices against the oracle,
    every slice against the constraint set."""
    torch.manual_seed(11)
    X = torch.randn(65536, 64).abs() + 1e-3
    n, sp = X.shape[0], 0.85
    L1 = n ** 0.5 * (1 - sp) + sp
    norms = hoy.get_norm(X)
    x = X.cuda()
    _engine.hoyer_project_(x, 1, (L1 * norms).cuda(), (norms * norms).cuda())
    y = x.cpu()
    assert float(y.min()) >= 0
    assert torch.allclose(y.sum(0), L1 * norms, rtol=1e-4)
    assert torch.allclose(hoy.get_norm(y), norms, rtol=1e-4)
    for j in (0, 17, 63):
        want = hoy.proj_func(X[:, j], float(L1 * norms[j]), float(norms[j] ** 2))
        assert _err(y[:, j], want, 1e-3, 1e-5) <= 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("name", SFIT)
def test_sparse_fit_matches_reference(name):
    c = _case(name)
    m = CLS[_kind(name)](W=_t(c, "W0"), H=_t(c, "H0"), trainable_W=bool(c["trainable_W"]),
                         trainable_H=bool(c["trainable_H"])).cuda()
    n_iter = m.sparse_fit(_t(c, "V").cuda(), float(c["beta"]), int(c["iters"]), False, _opt(c, "sW"), _opt(c, "sH"))
    assert n_iter == int(c["n_iter"])
    for got, want, nm in ((m.W.data.cpu(), _t(c, "W"), "W"), (m.H.data.cpu(), _t(c, "H"), "H")):
        e = _err(got, want, 1e-3, 1e-5)
        assert e <= 1.0, f"{name} {nm}: {e:.3f} x tolerance [{m.last_fit_precision}]"
    sW, sH = _opt(c, "sW"), _opt(c, "sH")
    if sH is not None and bool(c["trainable_H"]):                 # constraint set: every H component has sparseness sH, unit norm
        H = m.H.data.cpu()
        for r in range(H.shape[1]):
            assert float(sparseness(H[:, r])) == pytest.approx(sH, abs=2e-4)
        assert torch.allclose(hoy.get_norm(H), torch.ones(H.shape[1]), rtol=1e-4)
    if not bool(c["trainable_H"]):                                # (a frozen W is still rescaled by the renormalisation, nmf.py:588)
        assert torch.equal(m.H.data.cpu(), _t(c, "H0"))


@pytest.mark.gpu
def test_sparse_fit_host_buffers_and_sparse_target():
    """CPU-resident module and target are staged through the device; a sparse COO target gives the dense result."""
    c = _case("sfit_nmf_sW")
    V = _t(c, "V")
    m = NMF(W=_t(c, "W0"), H=_t(c, "H0"))
    m.sparse_fit(V, 2, int(c["iters"]), False, _opt(c, "sW"), None)
    assert m.W.device.type == "cpu"
    assert _err(m.W.data, _t(c, "W"), 1e-3, 1e-5) <= 1.0 and _err(m.H.data, _t(c, "H"), 1e-3, 1e-5) <= 1.0
    Vz = V * (V > 0.5)
    a = NMF(W=_t(c, "W0"), H=_t(c, "H0")).cuda()
    b = NMF(W=_t(c, "W0"), H=_t(c, "H0")).cuda()
    a.sparse_fit(Vz.cuda(), 2, 10, False, 0.5, 0.4)
    b.sparse_fit(Vz.to_sparse().cuda(), 2, 10, False, 0.5, 0.4)
    assert torch.equal(a.W.data, b.W.data) and torch.equal(a.H.data, b.H.data)


@pytest.mark.gpu
def test_unconstrained_sparse_fit_takes_the_tensor_core_path():
    """No constraint: multiplicative updates + renormalisation of H; precision "auto" keeps the fp16 tensor-core kernels."""
    torch.manual_seed(0)
    V = torch.rand(1024, 512).bfloat16().float()
    torch.manual_seed(1)
    W0, H0 = torch.randn(512, 32).abs(), torch.randn(1024, 32).abs()
    W, H, _, _ = hoy.sparse_fit(V, W0, H0, 1, 10)
    m = NMF(W=W0, H=H0).cuda()
    m.sparse_fit(V.cuda(), 1, 10)
    assert m.last_fit_precision == "f16"
    assert _err(m.W.data.cpu(), W, 1e-3, 1e-5) <= 1.0 and _err(m.H.data.cpu(), H, 1e-3, 1e-5) <= 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("name", SPROJ)
def test_sparsity_proj_matches_reference(name):
    c = _case(name)
    V = _t(c, "V").cuda()
    m = NMF(W=_t(c, "W0"), H=_t(c, "H0")).cuda()
    tr = SparsityProj([p for p, on in ((m.W, c["on_W"]), (m.H, c["on_H"])) if int(on)], float(c["sparsity"]))
    tr.param_groups[0]["lr"] = float(c["lr0"])

    def closure():
        tr.zero_grad()
        return beta_div(m(), V, float(c["beta"]))
    losses = [float(tr.step(closure)) for _ in range(int(c["steps"]))]
    assert tr.param_groups[0]["lr"] == pytest.approx(float(c["lr"]), rel=1e-12)
    assert np.allclose(losses, c["losses"], rtol=1e-4)
    assert _err(m.W.data.cpu(), _t(c, "W"), 1e-3, 1e-5) <= 1.0 and _err(m.H.data.cpu(), _t(c, "H"), 1e-3, 1e-5) <= 1.0
