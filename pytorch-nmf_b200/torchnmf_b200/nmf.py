"""NMF / NMFD modules with the reference's surface and a B200-native `fit`.

Mirrors the module surface of torchnmf 0.3.5 (`torchnmf/nmf.py`): `BaseComponent` (:173-292),
`NMF` (:641-697), `NMFD` (:700-779) and `BaseComponent.fit` (:298-409).  Constructor arguments,
parameter shapes (`W (C,R[,T])`, `H (N,R)` / `(B,R,L_in)`), `forward`, `state_dict` keys and the
`fit` signature / return value / exceptions are the reference's.  What differs is the inside of the
iteration loop: instead of materialising `WH` and taking two autograd backward passes
(`_double_backward_update`, :52-92), every update is one call into libnmf_b200.so, whose fused
sm_100a kernels never write the (N x C) reconstruction or ratio matrices to HBM.

There is no CPU compute path: `fit` on CPU-resident modules copies V / W / H to the current CUDA
device, runs there, and copies the factors back into the same Parameter storages ("host buffer"
mode, the `e2e` number of bench.py).  Without a CUDA device or without the built library it raises.

`NMF2D` (:782-865) and `NMF3D` (:868-942) run the NMFD contractions with the last axis sliding and the outer axes as loops.
Sparse targets are accepted by `NMF` (beta 1 / 2: the library's sparse kernels; other beta: densified on the device).
`sparse_fit` (:411-599, Hoyer's sparseness-constrained projected gradient) runs on the same engine: gradients from the fused
raw-terms launch, line-search losses from the fused loss launch, every component projected by ONE
`nmfb200_hoyer_project` launch.  `trainer.BetaMu` / `SparsityProj` and `plca.*` live in their own modules.
"""
import math
import weakref
from collections.abc import Iterable as _Iterable

import torch
import torch.nn.functional as F
from torch import Tensor
from torch.nn import Parameter

from .constants import eps  # noqa: F401  (re-exported like torchnmf.nmf does)
from . import engine as _engine

try:
    from tqdm import tqdm as _tqdm
except Exception:  # pragma: no cover
    _tqdm = None

__all__ = ["BaseComponent", "NMF", "NMFD", "NMF2D", "NMF3D"]


def _gamma(beta):
    # nmf.py:341-346
    if beta < 1:
        return 1.0 / (2.0 - beta)
    if beta > 2:
        return 1.0 / (beta - 1.0)
    return 1.0


def _get_norm(x, axis=1):
    """L2 norm over every axis but `axis` (nmf.py:134-139)."""
    dims = [d for d in range(x.dim()) if d != axis]
    return (x * x).sum(dims).sqrt()


@torch.no_grad()
def _renorm(W, H, unit_norm="W"):
    """Move the component norms to the other factor, in place (nmf.py:142-159)."""
    if unit_norm == "W":
        unit, other = W, H
    elif unit_norm == "H":
        unit, other = H, W
    else:
        raise ValueError("Input type isn't valid!")
    n = _get_norm(unit)
    unit /= n[(slice(None),) + (None,) * (unit.dim() - 2)]
    other *= n[(slice(None),) + (None,) * (other.dim() - 2)]


def _proj_func(s, k1, k2):
    """Hoyer's projection of ONE vector (any shape) onto {v >= 0, |v|_1 = k1, |v|_2^2 = k2} (nmf.py:21-49); returns a new
    tensor.  Runs in the library (`nmfb200_hoyer_project`): CUDA tensors only."""
    out = s.detach().clone().reshape(1, 1, -1)
    _engine.hoyer_project_(out, 1, [float(k1)], [float(k2)])
    return out.view(s.shape)


class _NullBar:
    def __init__(self, *a, **k): pass
    def __enter__(self): return self
    def __exit__(self, *a): return False
    def set_postfix(self, **k): pass
    def update(self, n): pass


class BaseComponent(torch.nn.Module):
    """Base class of the NMF modules (reference: nmf.py:173-292).

    Args:
        rank: size of the hidden dimension
        W / H: a size (iterable of ints -> random non-negative init) or an initial non-negative Tensor
        trainable_W / trainable_H: whether a *given tensor* is updated by `fit`
    """

    def __init__(self, rank=None, W=None, H=None, trainable_W=True, trainable_H=True):
        super().__init__()
        inferred = None
        for name, spec, trainable in (("W", W, trainable_W), ("H", H, trainable_H)):
            if isinstance(spec, Tensor):
                assert torch.all(spec >= 0.), f"Tensor {name} should be non-negative."   # nmf.py:215,227
                p = Parameter(torch.empty(*spec.size()), requires_grad=trainable)
                p.data.copy_(spec)
                self.register_parameter(name, p)
                inferred = p.shape[1]
            elif isinstance(spec, _Iterable):
                spec = tuple(spec)
                self.register_parameter(name, Parameter(torch.randn(*spec).abs()))       # nmf.py:221,234
                inferred = spec[1]
            else:
                self.register_parameter(name, None)

        if inferred is None:
            assert rank, "A rank should be given when W and H are not available!"        # nmf.py:240
        else:
            if self.H is not None:
                assert self.H.shape[1] == inferred, "Latent size of H does not match with others!"
            if self.W is not None:
                assert self.W.shape[1] == inferred, "Latent size of W does not match with others!"
                self.out_channels = self.W.shape[0]
                if self.W.ndim > 2:
                    self.kernel_size = self.W.shape[2:]
            rank = inferred
        self.rank = rank

    def extra_repr(self):
        s = f"{self.rank}"
        if self.W is not None:
            s += f", out_channels={self.out_channels}"
            if hasattr(self, "kernel_size"):
                s += f", kernel_size={tuple(self.kernel_size)}"
        return s

    def forward(self, H=None, W=None):
        """Reconstruction only (nmf.py:261-284); plain differentiable torch ops, not on the fit path."""
        own = H is None and W is None
        H = self.H if H is None else H
        W = self.W if W is None else W
        assert H is not None
        assert W is not None
        out = self.reconstruct(H, W)
        if own and type(self) in _BETAMU_FUSABLE:
            # the plain reconstruction of this module's own factors: lets trainer.BetaMu recognise a single-leaf graph
            # and take both update terms from the fused kernels instead of two backward passes through `out`
            out._nmf_b200_src = weakref.ref(self)
        return out

    @staticmethod
    def reconstruct(H, W):
        raise NotImplementedError

    # ---- engine selection -------------------------------------------------------------------
    _engine_cls = None

    def _build_engine(self, V, W, H, precision):
        return self._engine_cls(V, W, H, precision)

    def _check_target_shape(self, V):
        raise NotImplementedError

    # test hook (tests/oracle_engine.py): an engine class used instead of the CUDA engines, so the host logic of `fit`
    # can be tested on a GPU-less box.  Deliberately NOT a parameter of `fit`: its signature stays the reference's.
    _engine_factory = None
    _sparse_targets = False       # NMF only (nmf.py:603-638); the convolutive models raise, as in the reference
    _sparse_kernels = True        # beta 1 / 2 on a sparse target: the library's sparse kernels (False: densify)

    def _open_engine(self, V, beta, precision, group, sparse_kernels):
        """Shared entry of `fit` / `sparse_fit`: validation that needs no device pass, placement of V / W / H on the CUDA
        device (host buffers and other dtypes are staged through fp32 device copies) and the engine for this target.
        Returns (engine, W, H, Wd, Hd, staged): W / H the Parameters, Wd / Hd the fp32 device tensors the engine updates."""
        sparse_target = V.is_sparse
        if sparse_target and not self._sparse_targets:
            raise NotImplementedError                      # nmf.py:294-295: only NMF derives the sparse update
        if sparse_target:
            # The reference's sparse derivation (nmf.py:95-119, :603-638: SDDMM at the non-zeros) is the same update as the
            # dense one on V.to_dense() -- its own tests/test_nmf_sparse.py:8-37 asserts exactly that.  beta 1 and 2 run on
            # the library's sparse kernels (update terms at the non-zeros only, engine.CudaSparseNmfEngine); for any other
            # beta the reference itself forms WH densely (nmf.py:621-627), and so does this path: the target is densified
            # ON THE DEVICE and takes the fused dense kernels (memory = the dense size).  `sparse_kernels=False` forces that.
            V = V.coalesce()
            assert torch.all(V.values() >= 0.), "Target should be non-negative."            # nmf.py:329-330
            if beta <= 0:                                                                    # nmf.py:332-336
                raise ValueError("When beta <= 0 and V contains zeros, the training process may diverge. "
                                 "Please add small values to V, or use a positive beta value.")
        W, H = self.W, self.H
        assert W is not None and H is not None, "fit() needs both W and H"
        self._check_target_shape(V)

        # ---- placement: run on the parameters' CUDA device, or stage host buffers through cuda ----
        staged = False
        if self._engine_factory is None:
            if not torch.cuda.is_available():
                raise RuntimeError("torchnmf_b200.fit needs a CUDA device (sm_100a); there is no CPU fallback")
            f32 = torch.float32
            on_gpu = W.device.type == "cuda"
            dev = W.device if on_gpu else torch.device("cuda", torch.cuda.current_device())
            Vd = V.to(dev, non_blocking=True)
            use_sparse_kernels = (sparse_kernels and sparse_target and beta in (1, 2) and group is None
                                  and self._sparse_kernels)
            if not use_sparse_kernels:
                Vd = (Vd.to_dense() if sparse_target else Vd).to(f32).contiguous()
            if on_gpu and W.dtype == f32 and H.dtype == f32:
                Wd, Hd = W.data, H.data                       # updated in place, like param.data in the reference
            else:
                staged = True                                 # host buffers and / or another dtype: fp32 device copies
                Wd = W.data.to(dev, f32, non_blocking=True).contiguous()
                Hd = H.data.to(dev, f32, non_blocking=True).contiguous()
            if not Wd.is_contiguous() or not Hd.is_contiguous():
                raise ValueError("W and H must be contiguous")
            eng = (_engine.CudaSparseNmfEngine(Vd.coalesce(), Wd, Hd) if use_sparse_kernels
                   else self._build_engine(Vd, Wd, Hd, precision))
        else:
            Wd, Hd = W.data, H.data
            eng = self._engine_factory(V.to_dense() if (sparse_target and not sparse_kernels) else V, Wd, Hd)
        if group is not None:
            if eng.kind != "nmf":
                raise NotImplementedError("row sharding is implemented for NMF only (NMFD: replicas only)")
            eng = _engine.ShardedEngine(eng, group)
        return eng, W, H, Wd, Hd, staged

    @torch.no_grad()
    def fit(self, V, beta=1, tol=1e-4, max_iter=200, verbose=False, alpha=0, l1_ratio=0, *,
            precision="auto", group=None):
        """Learn the model for `V` by minimising the beta-divergence with multiplicative updates.

        Positional arguments, defaults, return value (`n_iter`) and exceptions are those of
        `BaseComponent.fit` in the reference (nmf.py:298-409).  Keyword-only extras:

        precision: "auto" | "f32" | "f16" | "f16_split" -- arithmetic of the contraction kernels ("auto": fp16
                   tensor-core operands where the target fits their range, fp32 CUDA cores otherwise)
        group:     a torch.distributed process group; V and H are then this rank's ROW shard
                   (rows of V <-> rows of H) and W is replicated; one all-reduce per W update.

        dtype: the kernels keep fp32 master factors and fp32 accumulators.  The reference computes in the module's
        dtype (nmf.py:214-218); here a float64 / half module (or target) is staged through fp32 copies and the result
        is written back into the same Parameter storages in their own dtype.
        """
        eng, W, H, Wd, Hd, staged = self._open_engine(V, beta, precision, group, sparse_kernels=True)

        try:
            vmin, vmax = eng.minmax()
            assert vmin >= 0., "Target should be non-negative."                            # nmf.py:329-330
            if vmin == 0 and beta <= 0:                                                    # nmf.py:332-336
                raise ValueError("When beta <= 0 and V contains zeros, the training process may diverge. "
                                 "Please add small values to V, or use a positive beta value.")
            gamma = _gamma(beta)
            l1_reg = alpha * l1_ratio                                                      # nmf.py:348
            l2_reg = alpha * (1 - l1_ratio)                                                # nmf.py:349

            def fit_loss(more=False):
                # `more`: a W update follows on these very factors -- the engine may take the loss out of that update's own
                # contraction pass (engine.loss_prefetch_w) instead of a pass over V of its own
                fold = more and hasattr(eng, "loss_prefetch_w")
                d = eng.loss_prefetch_w(beta) if fold else eng.loss(beta)
                return math.sqrt(2.0 * d) if d >= 0 else float("nan")                      # nmf.py:362,402

            loss_init = fit_loss()
            previous_loss = loss_init
            train_w, train_h = W.requires_grad, H.requires_grad
            bar = _tqdm(total=max_iter, disable=not verbose) if _tqdm is not None else _NullBar()
            n_iter = -1
            batched = train_w and train_h and group is None and hasattr(eng, "iterate")
            with bar as pbar:
                while batched and n_iter + 1 < max_iter:
                    # both factors trainable: run the iterations up to the next loss evaluation in one engine call
                    k = min(10 - ((n_iter + 1) % 10), max_iter - (n_iter + 1))
                    eng.iterate(k, beta, gamma, l1_reg, l2_reg)                            # nmf.py:366-391, k times
                    n_iter += k
                    if n_iter % 10 == 9:                                                   # nmf.py:393
                        loss = fit_loss(more=n_iter + 1 < max_iter)
                        pbar.set_postfix(loss=loss)
                        pbar.update(10)
                        if (previous_loss - loss) / loss_init < tol:                       # nmf.py:405
                            break
                        previous_loss = loss
                for n_iter in (range(max_iter) if not batched else ()):                    # nmf.py:366
                    if train_w:
                        eng.update_w(beta, gamma, l1_reg, l2_reg)                          # nmf.py:367-378
                    if train_h:
                        eng.update_h(beta, gamma, l1_reg, l2_reg)                          # nmf.py:380-391
                    if n_iter % 10 == 9:                                                   # nmf.py:393
                        loss = fit_loss(more=train_w and group is None and n_iter + 1 < max_iter)
                        pbar.set_postfix(loss=loss)
                        pbar.update(10)
                        if (previous_loss - loss) / loss_init < tol:                       # nmf.py:405
                            break
                        previous_loss = loss
            if hasattr(eng, "check_health"):
                eng.check_health()
            if staged:
                W.data.copy_(Wd)
                H.data.copy_(Hd)
            self.last_fit_precision = eng.precision_for(beta) if hasattr(eng, "precision_for") else eng.precision
            self.last_w_update_path = getattr(eng, "w_update_path", None)     # sharded fits: "peer" (NVLink P2P) or "nccl"
        finally:
            eng.close()
        return n_iter + 1                                                                  # nmf.py:409


    @torch.no_grad()
    def sparse_fit(self, V, beta=2, max_iter=200, verbose=False, sW=None, sH=None, *, precision="auto"):
        """Learn the model for `V` under Hoyer's sparseness constraints (reference: nmf.py:411-599).

        Positional arguments, defaults, return value and exceptions are the reference's: `sW` / `sH` in (0, 1) fix the
        sparseness of every component W[:, r] / H[:, r]; a factor without a constraint takes the multiplicative update
        (nmf.py:503-511), a constrained one a projected-gradient step with a halving line search (:513-538), and H is
        re-normalised to unit component norms after its update (:588).  No stop rule: `max_iter` iterations are run.

        On the engine: the gradient is `positive - negative` of ONE fused raw-terms launch (`nmfb200_*_raw_terms`), every
        line-search loss one fused loss launch on the trial factor, and the per-component Python loop around `_proj_func`
        (nmf.py:519-522: R x rounds x 7 ATen launches and one `.item()` per round) is one `nmfb200_hoyer_project` launch.

        precision: as in `fit`; "auto" resolves to "f32" when a constraint is active (the line search compares losses of
        nearly equal trial points).  Sparse targets are densified on the device.
        """
        constrained = ((sW is not None and self.W is not None and self.W.requires_grad)
                       or (sH is not None and self.H is not None and self.H.requires_grad))
        if precision == "auto" and constrained:
            precision = "f32"
        eng, W, H, Wd, Hd, staged = self._open_engine(V, beta, precision, None, sparse_kernels=False)
        try:
            vmin, vmax = eng.minmax()
            assert vmin >= 0., "Target should be non-negative."                            # nmf.py:447-448
            if vmin == 0 and beta <= 0:                                                    # nmf.py:450-454
                raise ValueError("When beta <= 0 and V contains zeros, the training process may diverge. "
                                 "Please add small values to V, or use a positive beta value.")
            train_w, train_h = W.requires_grad, H.requires_grad
            R = Wd.shape[1]
            L1a = L1s = None
            if sW is not None and train_w:                                                 # nmf.py:459-467
                L1a = Wd[:, 0].numel() ** 0.5 * (1 - sW) + sW
                eng.project(Wd, 1, [L1a] * R, [1.0] * R)
            if sH is not None and train_h:                                                 # nmf.py:469-477
                L1s = Hd[:, 0].numel() ** 0.5 * (1 - sH) + sH
                eng.project(Hd, 1, [L1s] * R, [1.0] * R)
            eng.sync()
            gamma = _gamma(beta)                                                           # nmf.py:479-484
            step = {0: 1.0, 1: 1.0}                                                        # nmf.py:490

            def projected_step(which, L1):
                """nmf.py:513-538 (W) / :559-586 (H): gradient step, projection of every component, halving line search."""
                cur = Wd if which == 0 else Hd
                loss = eng.loss(beta)
                num, den = eng.raw_terms(which, beta)
                if beta == 1:
                    den = den.view((1, -1) + (1,) * (cur.dim() - 2))                       # colsum of the other factor
                grad = den - num
                for _ in range(10):
                    new = cur - step[which] * grad
                    norms = _get_norm(new)
                    eng.project(new, 1, L1 * norms, norms * norms)
                    new_loss = eng.loss_at(new if which == 0 else Wd, Hd if which == 0 else new, beta)
                    if new_loss <= loss:
                        break
                    step[which] *= 0.5
                step[which] *= 1.2
                cur.copy_(new)
                eng.sync()

            bar = _tqdm(total=max_iter, disable=not verbose) if _tqdm is not None else _NullBar()
            n_iter = -1
            with bar as pbar:
                for n_iter in range(max_iter):
                    if train_w:
                        if L1a is None:
                            eng.update_w(beta, gamma, 0.0, 0.0)                            # nmf.py:503-511
                        else:
                            projected_step(0, L1a)
                    if train_h:
                        if L1s is None:
                            eng.update_h(beta, gamma, 0.0, 0.0)                            # nmf.py:549-557
                        else:
                            projected_step(1, L1s)
                        _renorm(Wd, Hd, "H")                                               # nmf.py:588
                        eng.sync()
                    if n_iter % 10 == 9 and verbose:                                       # nmf.py:590-598 (display only)
                        d = eng.loss(beta)
                        pbar.set_postfix(loss=math.sqrt(2.0 * d) if d >= 0 else float("nan"))
                        pbar.update(10)
            if hasattr(eng, "check_health"):
                eng.check_health()
            if staged:
                W.data.copy_(Wd)
                H.data.copy_(Hd)
            self.last_fit_precision = eng.precision_for(beta) if hasattr(eng, "precision_for") else eng.precision
        finally:
            eng.close()
        return n_iter + 1                                                                  # nmf.py:599


class NMF(BaseComponent):
    """Non-negative matrix factorisation  V (N,C) ~= H (N,R) @ W (C,R)^T   (reference: nmf.py:641-697)."""
    _engine_cls = _engine.CudaNmfEngine
    _sparse_targets = True

    def __init__(self, Vshape=None, rank=None, **kwargs):
        if isinstance(Vshape, _Iterable):
            M, K = Vshape                                  # wrong arity raises, as in the reference (:684)
            rank = rank if rank else K
            kwargs["W"] = (K, rank)
            kwargs["H"] = (M, rank)
        super().__init__(rank, **kwargs)

    @staticmethod
    def reconstruct(H, W):
        return F.linear(H, W)                              # H @ W^T, nmf.py:691-693

    def _check_target_shape(self, V):
        if V.dim() != 2 or V.shape[0] != self.H.shape[0] or V.shape[1] != self.W.shape[0]:
            raise RuntimeError(f"target shape {tuple(V.shape)} does not match H {tuple(self.H.shape)} / "
                               f"W {tuple(self.W.shape)}")


class NMFD(BaseComponent):
    """Non-negative matrix factor deconvolution (reference: nmf.py:700-779).

    V (B,C,L) ~= sum_t W[:,:,t] @ shift_t(H),  W (C,R,T), H (B,R,L-T+1).
    """
    _engine_cls = _engine.CudaNmfdEngine

    def __init__(self, Vshape=None, rank=None, T=1, **kwargs):
        if isinstance(Vshape, _Iterable):
            if isinstance(T, _Iterable):
                T, = T
            batch, K, M = Vshape                           # wrong arity raises, as in the reference (:769)
            rank = rank if rank else K
            kwargs["W"] = (K, rank, T)
            kwargs["H"] = (batch, rank, M - T + 1)
        super().__init__(rank, **kwargs)

    @staticmethod
    def reconstruct(H, W):
        return F.conv1d(H, W.flip(2), padding=W.shape[2] - 1)   # nmf.py:776-779

    def _check_target_shape(self, V):
        ok = (V.dim() == 3 and V.shape[0] == self.H.shape[0] and V.shape[1] == self.W.shape[0]
              and V.shape[2] == self.H.shape[2] + self.W.shape[2] - 1)
        if not ok:
            raise RuntimeError(f"target shape {tuple(V.shape)} does not match H {tuple(self.H.shape)} / "
                               f"W {tuple(self.W.shape)}")


def _ntuple(x, n):
    """torch.nn.modules.utils._pair / _triple: an int repeats, an iterable is taken as is."""
    return tuple(x) if isinstance(x, _Iterable) else (x,) * n


class _NMFnD(BaseComponent):
    """Shared part of NMF2D / NMF3D: V (B,C,*X) ~= sum over the kernel offsets t of W[:,:,t] @ shift_t(H),
    W (C,R,*kernel_size), H (B,R,*(X - kernel_size + 1)).  `fit` runs the same three sliding contractions as NMFD with the
    last axis sliding and the outer axes as loops (csrc/nmfd.cu), in fp32, for every beta."""
    _engine_cls = _engine.CudaNmfdEngine
    _nd = 0

    def _check_target_shape(self, V):
        nd = self._nd
        ok = (V.dim() == nd + 2 and V.shape[0] == self.H.shape[0] and V.shape[1] == self.W.shape[0]
              and all(V.shape[2 + i] == self.H.shape[2 + i] + self.W.shape[2 + i] - 1 for i in range(nd)))
        if not ok:
            raise RuntimeError(f"target shape {tuple(V.shape)} does not match H {tuple(self.H.shape)} / "
                               f"W {tuple(self.W.shape)}")


class NMF2D(_NMFnD):
    """Non-negative matrix factor 2-D deconvolution (reference: nmf.py:782-865).

    V (B,C,L,M) ~= conv2d(H, flipped W, full padding),  W (C,R,k0,k1),  H (B,R,L-k0+1,M-k1+1).
    """
    _nd = 2

    def __init__(self, Vshape=None, rank=None, kernel_size=1, **kwargs):
        if isinstance(Vshape, _Iterable):
            kernel_size = _ntuple(kernel_size, 2)
            kh, kw = kernel_size
            batch, channel, K, M = Vshape                  # wrong arity raises, as in the reference (:852)
            rank = rank if rank else K
            kwargs["W"] = (channel, rank) + kernel_size
            kwargs["H"] = (batch, rank, K - kh + 1, M - kw + 1)
        super().__init__(rank, **kwargs)

    @staticmethod
    def reconstruct(H, W):
        return F.conv2d(H, W.flip((2, 3)), padding=(W.shape[2] - 1, W.shape[3] - 1))          # nmf.py:861-865


class NMF3D(_NMFnD):
    """Non-negative matrix factor 3-D deconvolution (reference: nmf.py:868-942).

    V (B,C,N,K,M) ~= conv3d(H, flipped W, full padding),  W (C,R,k0,k1,k2),  H (B,R,N-k0+1,K-k1+1,M-k2+1).
    """
    _nd = 3

    def __init__(self, Vshape=None, rank=None, kernel_size=1, **kwargs):
        if isinstance(Vshape, _Iterable):
            kernel_size = _ntuple(kernel_size, 3)
            kd, kh, kw = kernel_size
            batch, channel, N, K, M = Vshape               # wrong arity raises, as in the reference (:928)
            rank = rank if rank else K
            kwargs["W"] = (channel, rank) + kernel_size
            kwargs["H"] = (batch, rank, N - kd + 1, K - kh + 1, M - kw + 1)
        super().__init__(rank, **kwargs)

    @staticmethod
    def reconstruct(H, W):
        pad = (W.shape[2] - 1, W.shape[3] - 1, W.shape[4] - 1)
        return F.conv3d(H, W.flip((2, 3, 4)), padding=pad)                                     # nmf.py:938-942


# module types whose plain reconstruction trainer.BetaMu may replace by the fused kernels (exact types: a subclass with its
# own `reconstruct` is a different model)
_BETAMU_FUSABLE = frozenset({NMF, NMFD, NMF2D, NMF3D})
