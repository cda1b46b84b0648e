"""Dense-NMF host paths of the C library that a single-GPU fit() does not reach, pinned so that the copies of them cannot drift
apart: the CUDA-core (f32) pieces of the row-sharded W update (w_partial -> sum -> w_apply), the CUDA-core raw terms,
w_partial as the W update's raw terms, and the error codes of the entry points.  Plus, without a GPU, which engine class
offers which optional operation: fit(), sparse_fit() and ShardedEngine pick their branch with hasattr."""
import ctypes

import pytest
import torch

from oracle import mu_oracle as orc
from torchnmf_b200 import _capi
from torchnmf_b200 import engine as _engine


def _close(a, b):
    """The suite's f32 tolerance (test_gpu_parity.py): rtol 2e-4, atol 1e-6 * max|b|."""
    return torch.allclose(a, b, rtol=2e-4, atol=1e-6 * float(b.abs().max()))


def _inputs(N, C, R, seed):
    torch.manual_seed(seed)
    return torch.rand(N, C) + 0.01, torch.rand(C, R) + 0.1, torch.rand(N, R) + 0.1


def _engine_on(V, W, H, precision):
    return _engine.CudaNmfEngine(V.cuda(), W.cuda(), H.cuda(), precision)


@pytest.mark.gpu
@pytest.mark.parametrize("beta", [0.5, 1, 2])
def test_f32_sharded_w_update_equals_the_full_w_update(beta):
    """Two row shards on one GPU: the sum of their w_partial buffers, applied by w_apply, is the W update of the whole target.
    R = 33 is not a multiple of 4 (the scalar ratio-stage kernel)."""
    N, C, R = 700, 300, 33
    V, W0, H0 = _inputs(N, C, R, 5)
    gamma, l1, l2 = orc.gamma_of(beta), 0.01, 0.02
    full = _engine_on(V, W0, H0, "f32")
    shards = [_engine_on(V[lo:hi], W0, H0[lo:hi], "f32") for lo, hi in ((0, 290), (290, N))]
    try:
        full.update_w(beta, gamma, l1, l2)
        reduced = shards[0].w_partial(beta) + shards[1].w_partial(beta)
        shards[1].w_apply(reduced, beta, gamma, l1, l2)
        assert shards[1].precision_for(beta) == "f32"
        assert _close(shards[1].W.cpu(), full.W.cpu())
    finally:
        for e in [full] + shards:
            e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("which", [0, 1])
@pytest.mark.parametrize("beta", [0, 1, 1.5, 2])
def test_f32_raw_terms_match_the_oracle_contractions(beta, which):
    """Numerator (rows, R) and denominator of one factor's update; for beta 1 the denominator is the other factor's column
    sum (R,)."""
    V, W0, H0 = _inputs(500, 260, 33, 6)
    eng = _engine_on(V, W0, H0, "f32")
    try:
        num, den = (t.cpu() for t in eng.raw_terms(which, beta))
    finally:
        eng.close()
    V, W, H = V.double(), W0.double(), H0.double()
    Pn, Pp = orc.phi(V, orc.nmf_reconstruct(H, W), beta)
    other = H if which == 0 else W
    want_num = (Pn.t() if which == 0 else Pn) @ other
    want_den = other.sum(0) if beta == 1 else (Pp.t() if which == 0 else Pp) @ other
    assert num.shape == want_num.shape and den.shape == want_den.shape
    assert _close(num, want_num.float()) and _close(den, want_den.float())


@pytest.mark.gpu
@pytest.mark.parametrize("precision, beta", [("f32", 0.5), ("f32", 1), ("f32", 2), ("f16", 1)])
def test_w_partial_is_the_w_raw_terms(precision, beta):
    """w_partial(beta) is raw_terms(0, beta) flattened (numerator, then denominator), bit for bit."""
    V, W0, H0 = _inputs(640, 384, 64, 7)
    eng = _engine_on(V, W0, H0, precision)
    try:
        assert eng.precision_for(beta) == precision
        num, den = eng.raw_terms(0, beta)
        want = torch.cat([num.reshape(-1), den.reshape(-1)])
        got = eng.w_partial(beta).clone()
    finally:
        eng.close()
    assert torch.equal(got, want)


@pytest.mark.gpu
def test_entry_points_return_their_error_codes():
    lib = _capi.load()
    N, C, R = 64, 48, 8
    torch.manual_seed(8)
    W, H = torch.rand(C, R, device="cuda"), torch.rand(N, R, device="cuda")
    out = torch.empty(2 * N * R, device="cuda")
    w, h, o = W.data_ptr(), H.data_ptr(), out.data_ptr()
    st = torch.cuda.current_stream().cuda_stream

    def call(fn, *args):
        return fn(*args), lib.nmfb200_last_error().decode()

    ctx = ctypes.c_void_p()
    _capi.check(lib.nmfb200_nmf_create(ctypes.byref(ctx), torch.cuda.current_device(), N, C, R, _capi.PREC_F32))
    try:
        assert call(lib.nmfb200_nmf_update_w, ctx, w, h, 1.0, 1.0, 0.0, 0.0, st) == (3, "set_target has not been called")
    finally:
        lib.nmfb200_destroy(ctx)

    V = torch.rand(N, C)
    V[V < 0.7] = 0
    eng = _engine.CudaSparseNmfEngine(V.to_sparse().cuda().coalesce(), W, H)
    try:
        sparse = (3, "not available for a sparse target")
        assert call(lib.nmfb200_nmf_raw_terms, eng._ctx, w, h, 0, 1.0, o, st) == sparse
        assert call(lib.nmfb200_nmf_raw_terms, eng._ctx, w, h, 1, 2.0, o, st) == sparse
        assert call(lib.nmfb200_nmf_w_partial, eng._ctx, w, h, 1.0, o, st) == sparse
        for fn in (lib.nmfb200_nmf_update_w, lib.nmfb200_nmf_update_h):
            rc, msg = call(fn, eng._ctx, w, h, 0.5, 1.0, 0.0, 0.0, st)
            assert rc == 1 and "beta must be 1 or 2" in msg
    finally:
        eng.close()


def test_optional_engine_operations_by_class():
    E = _engine
    classes = {E.CudaNmfEngine, E.CudaSparseNmfEngine, E.CudaNmfdEngine}

    def having(attr):
        return {c for c in classes if hasattr(c, attr)}

    assert having("iterate") == {E.CudaNmfEngine, E.CudaSparseNmfEngine}
    # defined in the class body itself: a test takes the folded loss away with monkeypatch.delattr on that class
    assert "loss_prefetch_w" in vars(E.CudaNmfEngine) and having("loss_prefetch_w") == {E.CudaNmfEngine}
    for attr in ("peer_supported", "w_partial", "w_apply", "contract_only"):
        assert having(attr) == {E.CudaNmfEngine}, attr
    for attr in ("precision_for", "check_health"):
        assert having(attr) == classes, attr
