"""Host-side engines: thin owners of an ``nmfb200_ctx`` plus the row-sharded W update.

An engine exposes exactly the operations ``BaseComponent.fit`` (nmf.py:366-407 in the reference)
needs from its loop body:

    minmax() -> (vmin, vmax)       fit()'s validation, nmf.py:329-336
    update_w / update_h            nmf.py:367-391
    loss(beta) -> float            metrics.beta_div of the current reconstruction, nmf.py:360-361,:400-401

`ShardedEngine` wraps any engine that also offers ``w_partial`` / ``w_apply`` / ``loss_tensor`` and
inserts the one collective per iteration that the row-sharded layout needs (SURVEY.md 8e).
"""
import ctypes
import os

import torch

from . import _capi


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def _stream(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _check_f32_cuda(t, name, device):
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32 (got {t.dtype}); the engine mirrors the reference's default dtype")
    if t.device != device:
        raise ValueError(f"{name} is on {t.device}, expected {device}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")


# Engine workspaces (the fp16 operand copies of V are the size of V) are kept across fit() calls of the same
# shape instead of being cudaMalloc'ed / cudaFree'd every time.  The memory is cudaMalloc'ed by the library, i.e. invisible
# to torch's caching allocator, so the cache is bounded by BYTES (estimated from the shapes): at most
# NMFB200_WORKSPACE_CACHE_MB (default 8192; 0 disables caching) are held between fits, in at most _MAX_WORKSPACES
# contexts.  release_workspaces() drops them all.
_WORKSPACES = {}
_MAX_WORKSPACES = 2
_CACHE_BYTES = int(float(os.environ.get("NMFB200_WORKSPACE_CACHE_MB", "8192")) * (1 << 20))


def _workspace_bytes(key):
    """Upper estimate of the device memory a cached context of this key holds."""
    if key[0] == "nmf":                   # ("nmf", device, N, C, R, precision): V16 + Vt16 + split partials + fp32 scratch
        _, _, N, C, R = key[:5]
        return 4 * N * C + 64 * (N + C) * max(R, 64)
    if key[0] == "nmfd":                  # ("nmfd", device, B, C, X, R, K, precision): ratio tiles + shifted operand copies
        _, _, B, C, X, R, K = key[:7]
        nx, nk = 1, 1
        for x in X:
            nx *= x
        for k in K:
            nk *= k
        return 12 * B * C * nx + 64 * C * R * nk + 64 * B * R * nx
    return 0


def cached_workspace_bytes():
    """Estimated device memory currently parked in the workspace cache."""
    return sum(_workspace_bytes(k) for k in _WORKSPACES)



def hoyer_project_(x, dim, k1, k2):
    """Project every slice of `x` along `dim` onto {v >= 0, |v|_1 = k1[j], |v|_2^2 = k2[j]} IN PLACE: ONE launch of
    `nmfb200_hoyer_project` (include/nmf_b200.h) for what the reference does with a Python loop over the slices around
    `_proj_func` (nmf.py:21-49, :519-522; trainer.py:176-181).  x: contiguous fp32 CUDA tensor; k1 / k2: sequences or
    tensors of x.shape[dim] values (device tensors are used as they are: no host synchronisation)."""
    if not (isinstance(x, torch.Tensor) and x.is_cuda):
        raise TypeError("hoyer_project_: x must be a CUDA tensor (the library has no CPU path)")
    if x.dtype != torch.float32 or not x.is_contiguous():
        raise TypeError("hoyer_project_: x must be a contiguous float32 tensor")
    D = x.shape[dim]
    outer = 1
    for n in x.shape[:dim]:
        outer *= n
    inner = x.numel() // max(outer * D, 1)
    if x.numel() == 0:
        return x
    k1 = torch.as_tensor(k1, dtype=torch.float32, device=x.device).contiguous()
    k2 = torch.as_tensor(k2, dtype=torch.float32, device=x.device).contiguous()
    assert k1.numel() == D and k2.numel() == D
    zeroed = torch.empty(x.numel(), dtype=torch.uint8, device=x.device)
    lib = _capi.load()
    _capi.check(lib.nmfb200_hoyer_project(x.device.index if x.device.index is not None else torch.cuda.current_device(),
                                          _ptr(x), outer, D, inner, _ptr(k1), _ptr(k2), _ptr(zeroed), _stream(x.device)))
    return x


def release_workspaces():
    """Free every cached engine workspace (device memory held between fit() calls)."""
    lib = _capi.load()
    for ctx in _WORKSPACES.values():
        lib.nmfb200_destroy(ctx)
    _WORKSPACES.clear()


class _CudaEngine:
    kind = None          # "nmf" or "nmfd": the family of nmfb200_<kind>_* entry points the engine calls

    def __init__(self):
        self._lib = _capi.load()
        self._ctx = ctypes.c_void_p()
        self._loss = None
        self._key = None
        self._wbuf = None

    def _acquire(self, key, create):
        """Take a cached context for `key` or create one with `create(ctx_ref)`."""
        self._key = key
        ctx = _WORKSPACES.pop(key, None)
        if ctx is not None:
            self._ctx = ctx
            return
        _capi.check(create(ctypes.byref(self._ctx)))

    def close(self):
        if self._ctx:
            mine = _workspace_bytes(self._key) if self._key is not None else 0
            if self._key is not None and mine <= _CACHE_BYTES:
                while _WORKSPACES and (len(_WORKSPACES) >= _MAX_WORKSPACES
                                       or cached_workspace_bytes() + mine > _CACHE_BYTES):
                    old = _WORKSPACES.pop(next(iter(_WORKSPACES)))
                    self._lib.nmfb200_destroy(old)
                _WORKSPACES[self._key] = self._ctx
            else:
                self._lib.nmfb200_destroy(self._ctx)
            self._ctx = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def _dev_index(self):
        return self.device.index if self.device.index is not None else torch.cuda.current_device()

    def _call(self, name, *args):
        """nmfb200_<kind>_<name>(ctx, *args, stream) on the engine's current stream; raises on an error code."""
        _capi.check(getattr(self._lib, f"nmfb200_{self.kind}_{name}")(self._ctx, *args, _stream(self.device)))

    def update_w(self, beta, gamma, l1_reg, l2_reg):
        self._call("update_w", _ptr(self.W), _ptr(self.H), beta, gamma, l1_reg, l2_reg)

    def update_h(self, beta, gamma, l1_reg, l2_reg):
        self._call("update_h", _ptr(self.W), _ptr(self.H), beta, gamma, l1_reg, l2_reg)

    def loss_tensor(self, beta):
        self._call("loss", _ptr(self.W), _ptr(self.H), beta, _ptr(self._loss))
        return self._loss

    def raw_terms(self, which, beta):
        """(numerator, denominator) of the update of W (which=0) or H (which=1) from the CURRENT factors, untouched, in
        the factor's own shape; the denominator is (R,) for beta == 1 (the column sums of the other factor).  What
        BetaMu.step, PLCA.fit and sparse_fit are built from (include/nmf_b200.h: nmfb200_nmf_raw_terms, _nmfd_raw_terms)."""
        f = self.W if which == 0 else self.H
        n = int(getattr(self._lib, f"nmfb200_{self.kind}_raw_terms_numel")(self._ctx, int(which), float(beta)))
        buf = torch.empty(n, dtype=torch.float32, device=self.device)
        self._call("raw_terms", _ptr(self.W), _ptr(self.H), int(which), float(beta), _ptr(buf))
        num, den = buf[:f.numel()].view(f.shape), buf[f.numel():]
        return num, (den if beta == 1 else den.view(f.shape))

    @property
    def precision(self):
        return _capi.PRECISION_NAMES[self._lib.nmfb200_precision(self._ctx)]

    def precision_for(self, beta):
        """Arithmetic the contraction kernels use for this beta ("f32" when the tensor-core path does not cover it)."""
        return _capi.PRECISION_NAMES[self._lib.nmfb200_precision_for_beta(self._ctx, float(beta))]

    def minmax(self):
        vmin, vmax = ctypes.c_float(), ctypes.c_float()
        _capi.check(self._lib.nmfb200_target_minmax(self._ctx, ctypes.byref(vmin), ctypes.byref(vmax),
                                                    _stream(self.device)))
        return vmin.value, vmax.value

    def loss(self, beta):
        val = float(self.loss_tensor(beta).item())
        self.check_health()
        return val

    def check_health(self):
        """Raise if a kernel of the library aborted an internal wait since the last check (synchronises)."""
        _capi.check(self._lib.nmfb200_ctx_check_health(self._ctx, _stream(self.device)))

    # ---- what sparse_fit (nmf.py:411-599) needs beyond the MU updates ----
    def project(self, x, dim, k1, k2):
        """Hoyer projection of every slice of x along `dim`, in place (one launch)."""
        return hoyer_project_(x, dim, k1, k2)

    def loss_at(self, W, H, beta):
        """beta-divergence of the reconstruction from TRIAL factors (same shapes as the engine's own; a line search's
        candidate).  The engine's operand copies follow the trial factors: call sync() after committing or discarding."""
        keep = self.W, self.H
        self.W, self.H = W, H
        try:
            self.sync()
            return self.loss(beta)
        finally:
            self.W, self.H = keep


class _NmfEngine(_CudaEngine):
    """What the dense and the sparse-target NMF engines share beyond _CudaEngine."""
    kind = "nmf"

    def iterate(self, n_iter, beta, gamma, l1_reg, l2_reg):
        """n_iter x (update_w; update_h) in one host call."""
        self._call("iterate", _ptr(self.W), _ptr(self.H), beta, gamma, l1_reg, l2_reg, int(n_iter))


class CudaNmfEngine(_NmfEngine):
    """Dense NMF on one GPU: V (N,C), W (C,R), H (N,R), all fp32 CUDA tensors (W, H updated in place)."""

    def __init__(self, V, W, H, precision="auto"):
        super().__init__()
        self.device = W.device
        for t, n in ((V, "V"), (W, "W"), (H, "H")):
            _check_f32_cuda(t, n, self.device)
        N, C = V.shape
        R = W.shape[1]
        assert W.shape == (C, R) and H.shape == (N, R)
        self.V, self.W, self.H = V, W, H
        self.N, self.C, self.R = N, C, R
        dev_index = self._dev_index
        self._acquire(("nmf", dev_index, N, C, R, precision),
                      lambda ref: self._lib.nmfb200_nmf_create(ref, dev_index, N, C, R, _capi.PRECISIONS[precision]))
        self._loss = torch.zeros(1, dtype=torch.float64, device=self.device)
        _capi.check(self._lib.nmfb200_nmf_set_target(self._ctx, _ptr(V), V.stride(0), _stream(self.device)))
        self.sync()

    def sync(self):
        _capi.check(self._lib.nmfb200_nmf_sync_factors(self._ctx, _ptr(self.W), _ptr(self.H), _stream(self.device)))

    def loss_prefetch_w(self, beta):
        """The loss at the current factors, taken out of the NEXT W update's contraction pass where the library can fold it
        (beta 1 on the tensor-core path): that update then skips its contraction.  Same value as loss() (synchronises)."""
        _capi.check(self._lib.nmfb200_nmf_loss_prefetch_w(self._ctx, _ptr(self.W), _ptr(self.H), beta, _ptr(self._loss),
                                                          _stream(self.device)))
        val = float(self._loss.item())
        self.check_health()
        return val

    def contract_only(self, which, beta):
        """bench.py: launch only the fused contraction kernel (0 = W update's, 1 = H update's)."""
        _capi.check(self._lib.nmfb200_nmf_contract_only(self._ctx, _ptr(self.W), _ptr(self.H), which, beta,
                                                        _stream(self.device)))

    # --- pieces of the row-sharded W update -------------------------------------------------
    def w_partial(self, beta):
        n = int(self._lib.nmfb200_nmf_w_partial_numel(self._ctx, beta))
        buf = self._wbuf
        if buf is None or buf.numel() != n:           # one buffer per engine, reused every iteration
            buf = self._wbuf = torch.empty(n, dtype=torch.float32, device=self.device)
        _capi.check(self._lib.nmfb200_nmf_w_partial(self._ctx, _ptr(self.W), _ptr(self.H), beta, _ptr(buf),
                                                    _stream(self.device)))
        return buf

    # ---- row-sharded W update over peer memory (include/nmf_b200.h: nmfb200_nmf_peer_*) ----
    def peer_supported(self, beta):
        return bool(self._lib.nmfb200_nmf_peer_supported(self._ctx, float(beta)))

    def peer_world(self):
        return int(self._lib.nmfb200_nmf_peer_world(self._ctx))

    def peer_alloc(self):
        h = (ctypes.c_ubyte * 64)()
        _capi.check(self._lib.nmfb200_nmf_peer_alloc(self._ctx, ctypes.cast(h, ctypes.c_void_p)))
        return bytes(h)

    def peer_connect(self, world, rank, handles):
        buf = (ctypes.c_ubyte * (64 * world)).from_buffer_copy(handles)
        return int(self._lib.nmfb200_nmf_peer_connect(self._ctx, int(world), int(rank), ctypes.cast(buf, ctypes.c_void_p)))

    def peer_release(self):
        self._lib.nmfb200_nmf_peer_release(self._ctx)

    def update_w_peer(self, beta, gamma, l1_reg, l2_reg):
        _capi.check(self._lib.nmfb200_nmf_update_w_peer(self._ctx, _ptr(self.W), _ptr(self.H), beta, gamma, l1_reg,
                                                        l2_reg, _stream(self.device)))

    def w_apply(self, reduced, beta, gamma, l1_reg, l2_reg):
        _capi.check(self._lib.nmfb200_nmf_w_apply(self._ctx, _ptr(self.W), _ptr(reduced), beta, gamma, l1_reg,
                                                  l2_reg, _stream(self.device)))


class CudaSparseNmfEngine(_NmfEngine):
    """NMF on a sparse target, beta 1 or 2 (reference: nmf.py:603-638): V is a coalesced sparse COO tensor (N,C) on the device;
    its CSR and CSC forms are built here with torch (data-format plumbing) and the update terms are evaluated at the non-zeros
    only by the library (include/nmf_b200.h: nmfb200_nmf_set_target_sparse)."""

    def __init__(self, V, W, H, precision="auto"):
        super().__init__()
        self.device = W.device
        for t, n in ((W, "W"), (H, "H")):
            _check_f32_cuda(t, n, self.device)
        assert V.is_sparse and V.is_coalesced() and V.device == W.device
        N, C = V.shape
        R = W.shape[1]
        assert W.shape == (C, R) and H.shape == (N, R)
        self.W, self.H = W, H
        vals = V.values().to(torch.float32).contiguous()
        rows, cols = V.indices()[0].contiguous(), V.indices()[1].contiguous()      # coalesced: sorted by (row, col)
        nnz = int(vals.numel())
        self._crow = torch.zeros(N + 1, dtype=torch.int64, device=self.device)
        self._crow[1:] = torch.cumsum(torch.bincount(rows, minlength=N), 0)
        order = torch.argsort(cols * N + rows)                                     # the same entries sorted by (col, row)
        self._ccol = torch.zeros(C + 1, dtype=torch.int64, device=self.device)
        self._ccol[1:] = torch.cumsum(torch.bincount(cols, minlength=C), 0)
        self._col, self._val = cols, vals
        self._row, self._val_t = rows[order].contiguous(), vals[order].contiguous()
        v64 = vals.double()
        pos = v64[v64 > 0]
        self._vnorm_kl = float((pos * pos.log()).sum() - v64.sum())                # nmf.py:166-167 (0 log 0 = 0)
        self._vnorm_eu = float((v64 * v64).sum() * 0.5)                            # nmf.py:164-165
        self._vmin = float(vals.min()) if nnz else 0.0
        self._vmax = float(vals.max()) if nnz else 0.0
        self._has_zeros = nnz < N * C
        dev_index = self._dev_index
        self._acquire(("nmf", dev_index, N, C, R, "f32"),
                      lambda ref: self._lib.nmfb200_nmf_create(ref, dev_index, N, C, R, _capi.PRECISIONS["f32"]))
        self._loss = torch.zeros(1, dtype=torch.float64, device=self.device)
        _capi.check(self._lib.nmfb200_nmf_set_target_sparse(
            self._ctx, nnz, _ptr(self._crow), _ptr(self._col), _ptr(self._val), _ptr(self._ccol), _ptr(self._row),
            _ptr(self._val_t), self._vnorm_kl, self._vnorm_eu, _stream(self.device)))

    @property
    def precision(self):
        return "f32"

    def precision_for(self, beta):
        return "f32"

    def minmax(self):
        return (min(self._vmin, 0.0) if self._has_zeros else self._vmin), self._vmax

    def sync(self):
        pass


class CudaNmfdEngine(_CudaEngine):
    """NMFD / NMF2D / NMF3D on one GPU: V (B,C,*X), W (C,R,*K), H (B,R,*(X-K+1)) over one to three convolved axes."""
    kind = "nmfd"

    def __init__(self, V, W, H, precision="auto"):
        super().__init__()
        self.device = W.device
        for t, n in ((V, "V"), (W, "W"), (H, "H")):
            _check_f32_cuda(t, n, self.device)
        B, C, *X = V.shape
        _, R, *K = W.shape
        nd = len(X)
        assert 1 <= nd <= 3 and len(K) == nd
        assert W.shape == (C, R, *K) and H.shape == (B, R, *(x - k + 1 for x, k in zip(X, K)))
        self.V, self.W, self.H = V, W, H
        dev_index = self._dev_index
        if nd == 1:
            create = lambda ref: self._lib.nmfb200_nmfd_create(ref, dev_index, B, C, X[0], R, K[0],
                                                               _capi.PRECISIONS[precision])
        else:
            if precision not in ("auto", "f32"):
                raise ValueError("NMF2D / NMF3D run on the fp32 kernels: precision must be 'auto' or 'f32'")
            vd, kd = (ctypes.c_int64 * nd)(*X), (ctypes.c_int64 * nd)(*K)
            create = lambda ref: self._lib.nmfb200_nmfnd_create(ref, dev_index, B, C, nd, vd, R, kd,
                                                                _capi.PRECISIONS[precision])
        self._acquire(("nmfd", dev_index, B, C, tuple(X), R, tuple(K), precision), create)
        self._loss = torch.zeros(1, dtype=torch.float64, device=self.device)
        _capi.check(self._lib.nmfb200_nmfd_set_target(self._ctx, _ptr(V), _stream(self.device)))

    def sync(self):
        _capi.check(self._lib.nmfb200_nmfd_sync_factors(self._ctx))


class ShardedEngine:
    """Row-sharded NMF over a process group: every rank holds V[n_g,:], H[n_g,:] and a replica of W.

    H update and phi stage are local.  The W update is `local raw contraction -> ONE sum-all-reduce ->
    identical ratio stage on every rank` (relu/eps/l1/l2/gamma are applied after the reduction because
    they are not linear).  The loss is one more scalar all-reduce every 10th iteration, and min/max
    for validation one at entry.  No V or H data ever moves.
    """

    def __init__(self, local, group=None):
        import torch.distributed as dist
        self._dist = dist
        self.local = local
        self.group = group
        self.kind = local.kind
        self.world = dist.get_world_size(group)
        self._peer = {}                      # beta -> does the W update run over peer memory
        self.w_update_path = "nccl"

    @property
    def precision(self):
        return self.local.precision

    def precision_for(self, beta):
        return self.local.precision_for(beta) if hasattr(self.local, "precision_for") else self.local.precision

    def close(self):
        self.local.close()

    def sync(self):
        self.local.sync()

    def minmax(self):
        vmin, vmax = self.local.minmax()
        t = torch.tensor([-vmin, vmax], dtype=torch.float32, device=self._reduce_device())
        if vmin != vmin or vmax != vmax:          # NaN must survive the reduction
            t.fill_(float("nan"))
        self._dist.all_reduce(t, op=self._dist.ReduceOp.MAX, group=self.group)
        t = t.cpu()
        return -float(t[0]), float(t[1])

    def _reduce_device(self):
        dev = getattr(self.local, "device", None)
        return dev if dev is not None else torch.device("cpu")

    def _peer_ready(self, beta):
        """Collective, once per (engine, beta): may the W update run over peer memory?  Every rank must answer the same, so
        each step is agreed with a MIN all-reduce.  Off with NMFB200_PEER=0, on another backend than NCCL, beyond 8 ranks, or
        when the CUDA IPC handles cannot be opened (ranks on different nodes): the NCCL all-reduce path is used then."""
        key = float(beta)
        if key in self._peer:
            return self._peer[key]
        dist, loc = self._dist, self.local
        ok = (os.environ.get("NMFB200_PEER", "1") != "0" and hasattr(loc, "peer_supported") and 2 <= self.world <= 8
              and dist.get_backend(self.group) == "nccl" and loc.peer_supported(beta))
        dev = self._reduce_device()
        connected = bool(ok) and loc.peer_world() == self.world
        t = torch.tensor([int(bool(ok)), int(connected)], dtype=torch.int32, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN, group=self.group)
        ok, connected = bool(t[0].item()), bool(t[1].item())
        if ok and not connected:
            mine = torch.frombuffer(bytearray(loc.peer_alloc()), dtype=torch.uint8).to(dev)
            allh = torch.empty(self.world * 64, dtype=torch.uint8, device=dev)
            dist.all_gather_into_tensor(allh, mine, group=self.group)
            rc = loc.peer_connect(self.world, dist.get_rank(self.group), allh.cpu().numpy().tobytes())
            t = torch.tensor([int(rc == 0)], dtype=torch.int32, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN, group=self.group)
            ok = bool(t[0].item())
            if not ok:
                loc.peer_release()
        self._peer[key] = ok
        self.w_update_path = "peer" if ok else "nccl"
        return ok

    def update_w(self, beta, gamma, l1_reg, l2_reg):
        if self._peer_ready(beta):
            self.local.update_w_peer(beta, gamma, l1_reg, l2_reg)     # contraction -> publish -> fused P2P sum + ratio stage
            return
        buf = self.local.w_partial(beta)
        self._dist.all_reduce(buf, op=self._dist.ReduceOp.SUM, group=self.group)
        self.local.w_apply(buf, beta, gamma, l1_reg, l2_reg)

    def update_h(self, beta, gamma, l1_reg, l2_reg):
        self.local.update_h(beta, gamma, l1_reg, l2_reg)

    def loss(self, beta):
        t = self.local.loss_tensor(beta).clone()
        self._dist.all_reduce(t, op=self._dist.ReduceOp.SUM, group=self.group)
        val = float(t.item())
        self.check_health()
        return val

    def check_health(self):
        if hasattr(self.local, "check_health"):
            self.local.check_health()
