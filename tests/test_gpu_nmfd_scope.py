"""Which NMFD shapes run on the tensor-core kernels (csrc/tc_nmfd.cu): those of at most 128 shifts, the extent of wgrad's
single accumulator.  Module surface -> ctypes -> C ABI, against the oracle's fit (oracle/mu_oracle.py) at the north-star
tolerance: rtol 1e-3, atol 1e-5 * max|factor|."""
import pytest
import torch

from oracle import mu_oracle as orc
from torchnmf_b200 import NMFD
from torchnmf_b200._capi import NmfB200Error

pytestmark = pytest.mark.gpu
B, C, L, R = 1, 96, 700, 4


def _inputs(T, seed=0):
    torch.manual_seed(seed)
    return torch.rand(B, C, L), torch.rand(C, R, T) + 0.1, torch.rand(B, R, L - T + 1) + 0.1


def _close(got, want, rtol=1e-3, atol_rel=1e-5):
    atol = atol_rel * float(want.abs().max())
    return ((got - want).abs() / (rtol * want.abs() + atol)).max().item()


@pytest.mark.parametrize("T, want", [(128, "f16"), (129, "f32"), (160, "f32")])
def test_auto_runs_tensor_cores_up_to_128_shifts(T, want):
    V, W0, H0 = _inputs(T)
    m = NMFD(W=W0, H=H0).cuda()
    m.fit(V.cuda(), 1, float("-inf"), 2)
    assert m.last_fit_precision == want


def test_long_kernel_fit_matches_oracle():
    """T = 160 used to run on the tensor cores, whose wgrad computes shifts t < 128 only: the W numerator of the longer
    shifts was whatever the partial buffer held.  `auto` now runs it on the fp32 kernels."""
    T = 160
    V, W0, H0 = _inputs(T, seed=1)
    W, H, n_ref, _ = orc.fit(V.double(), W0.double(), H0.double(), beta=1, tol=float("-inf"), max_iter=10, kind="nmfd")
    m = NMFD(W=W0, H=H0).cuda()
    n = m.fit(V.cuda(), 1, float("-inf"), 10)
    assert n == n_ref == 10
    for got, want, nm in ((m.W.data.cpu().double(), W, "W"), (m.H.data.cpu().double(), H, "H")):
        err = _close(got, want)
        assert err <= 1.0, f"{nm} [{m.last_fit_precision}]: {err:.2f} x tolerance"


def test_f16_rejects_kernels_longer_than_128_shifts():
    V, W0, H0 = _inputs(160)
    m = NMFD(W=W0, H=H0).cuda()
    with pytest.raises(NmfB200Error, match="T <= 128"):
        m.fit(V.cuda(), 1, float("-inf"), 1, precision="f16")


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_tensor_core_fits_on_two_devices_in_one_process():
    """The kernels' shared-memory limits (about 110 KB per CTA at T = 128) are per-device state: a context on a second
    device must set them there too."""
    V, W0, H0 = _inputs(128, seed=2)
    out = []
    for dev in ("cuda:0", "cuda:1"):
        m = NMFD(W=W0, H=H0).to(dev)
        m.fit(V.to(dev), 1, float("-inf"), 5)
        assert m.last_fit_precision == "f16"
        out.append((m.W.data.cpu(), m.H.data.cpu()))
    assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1])
