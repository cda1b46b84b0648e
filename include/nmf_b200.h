/*
 * nmf_b200.h -- C ABI of the B200-native multiplicative-update NMF engine (libnmf_b200.so).
 *
 * This is the drop-in boundary for ONE hot path of yoyololicon/pytorch-NMF (torchnmf 0.3.5):
 * the body of BaseComponent.fit()'s iteration loop for dense targets
 *
 *     torchnmf/nmf.py:366-407   for n_iter in range(max_iter): W update, H update, loss every 10th
 *
 * i.e. reconstruct (nmf.py:691-693 NMF, :776-779 NMFD) + _double_backward_update (nmf.py:52-92)
 * + the KL denominators (nmf.py:122-131) + metrics.beta_div (metrics.py:60-96).  The reference has
 * no FFI: its seam is Python (SURVEY.md 8b).  The binding a maintainer adds on the reference side is
 * the ctypes stub shown in INTEGRATION.md; the Python host side shipped here
 * (pytorch-nmf_b200/torchnmf_b200) is that stub plus the unchanged NMF/NMFD module surface.
 *
 * Conventions
 *   - plain C: pointers, sizes, doubles.  No torch / C++ types.
 *   - all matrix pointers are DEVICE pointers to fp32, row-major, reference layout:
 *       NMF : V (N,C)   W (C,R)   H (N,R)            V ~= H @ W^T            (nmf.py:659-662)
 *       NMFD: V (B,C,L) W (C,R,T) H (B,R,L-T+1)      V ~= conv1d(H, flip(W)) (nmf.py:743-750)
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).  Every call is
 *     asynchronous on that stream unless documented as synchronising.
 *   - W / H are the caller's storages (the nn.Parameter .data of the reference); updates are
 *     performed IN PLACE on them (nmf.py:92).  V is borrowed read-only.
 *   - every function returns 0 on success; on failure a non-zero code, and
 *     nmfb200_last_error() describes it.  There is no CPU fallback anywhere in this library.
 */
#ifndef NMF_B200_H_
#define NMF_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NMFB200_ABI_VERSION 1

/* arithmetic mode of the contraction kernels */
enum {
  NMFB200_PREC_AUTO      = -1, /* f16 tensor-core path when the rank allows it (R <= 128), else f32 */
  NMFB200_PREC_F32       = 0,  /* fused CUDA-core kernels, fp32 operands and accumulators (exact) */
  NMFB200_PREC_F16       = 1,  /* tcgen05, fp16 operands, fp32 accumulate                         */
  NMFB200_PREC_F16_SPLIT = 2   /* tcgen05, fp16 hi/lo split factors (~22-bit), fp16 ratio tile    */
};

/* error codes */
enum {
  NMFB200_OK = 0,
  NMFB200_ERR_INVALID = 1,     /* bad argument / unsupported shape for the requested mode */
  NMFB200_ERR_CUDA = 2,        /* CUDA runtime / driver error                             */
  NMFB200_ERR_STATE = 3        /* call order violated (e.g. update before set_target)     */
};

typedef struct nmfb200_ctx nmfb200_ctx;

int         nmfb200_abi_version(void);
const char* nmfb200_last_error(void);
/* "src=<sha256/16 of csrc/* + this header> nvcc=<version> arch=sm_100a built=<date time>": which sources this binary is */
const char* nmfb200_build_info(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
int64_t     nmfb200_launch_count(void);

/* Synchronises `stream` and reports whether any kernel of this library aborted an internal wait (a protocol
 * bug or a wedged device): 0 = healthy, non-zero = the results since the last check are invalid. */
int nmfb200_check_health(void* stream);
/* Same, on the context's device (the plain form looks at whichever device is current); the caller's current device is
 * left unchanged, as it is by every entry point that takes a context. */
int nmfb200_ctx_check_health(nmfb200_ctx* ctx, void* stream);

/* ---- dense NMF ------------------------------------------------------------------------- */

/* Allocate the engine workspace for an (N,C) target of rank R on CUDA device `device`.
 * Mirrors the sizes fixed by NMF.__init__ (nmf.py:679-689). */
int nmfb200_nmf_create(nmfb200_ctx** out, int device, int64_t N, int64_t C, int64_t R, int precision);
void nmfb200_destroy(nmfb200_ctx* ctx);
/* which NMFB200_PREC_* the context resolved to */
int nmfb200_precision(const nmfb200_ctx* ctx);
/* which NMFB200_PREC_* the contraction kernels use for this beta (the tensor-core path covers beta != 2 for
 * rank <= 64 and beta == 1 for rank <= 128; everything else runs the fp32 kernels) */
int nmfb200_precision_for_beta(const nmfb200_ctx* ctx, double beta);

/* Register the target V (device fp32, leading dimension ldv >= C).  Builds the engine-private
 * operand copies and the V-only loss terms.  Replaces nothing in the reference: V is simply the
 * argument of fit() (nmf.py:299).  Asynchronous. */
int nmfb200_nmf_set_target(nmfb200_ctx* ctx, const float* V, int64_t ldv, void* stream);
/* min / max of the registered target (fit()'s validation, nmf.py:329-336).  Synchronises. */
int nmfb200_target_minmax(nmfb200_ctx* ctx, float* vmin, float* vmax, void* stream);

/* Tell the engine the fp32 factors changed outside its own update calls (fit() entry,
 * load_state_dict, a frozen factor): rebuilds operand copies and column sums.  Asynchronous. */
int nmfb200_nmf_sync_factors(nmfb200_ctx* ctx, const float* W, const float* H, void* stream);

/* One W update, nmf.py:367-378:  W <- W * ((relu(Pn^T H)+eps) / den)^gamma  in place.
 * l1_reg / l2_reg as computed at nmf.py:348-349; gamma as nmf.py:341-346. */
int nmfb200_nmf_update_w(nmfb200_ctx* ctx, float* W, const float* H,
                         double beta, double gamma, double l1_reg, double l2_reg, void* stream);
/* One H update with the current (already updated) W, nmf.py:380-391. */
int nmfb200_nmf_update_h(nmfb200_ctx* ctx, const float* W, float* H,
                         double beta, double gamma, double l1_reg, double l2_reg, void* stream);
/* n_iter consecutive MU iterations with both factors trainable: exactly n_iter x (update_w; update_h), i.e.
 * nmf.py:366-391 repeated, in one host call. */
int nmfb200_nmf_iterate(nmfb200_ctx* ctx, float* W, float* H, double beta, double gamma, double l1_reg,
                        double l2_reg, int n_iter, void* stream);
/* beta_div(H W^T, V, beta) (metrics.py:60-96) accumulated into the DEVICE double *loss_dev
 * (one element, overwritten).  Row shards add: the sum over ranks is the global divergence. */
int nmfb200_nmf_loss(nmfb200_ctx* ctx, const float* W, const float* H, double beta,
                     double* loss_dev, void* stream);
/* The same value, evaluated at the factors the NEXT W update starts from (nmf.py:393-402 runs right before nmf.py:367 of the
 * following iteration): on the tensor-core path for beta == 1 the loss sums come out of the W update's own contraction pass
 * (one lg2 per element on the S tile that pass forms anyway, instead of a pass over V of its own), and the next
 * nmfb200_nmf_update_w / nmfb200_nmf_iterate on UNCHANGED factors with the same beta skips its contraction.  Any other
 * call in between (or a stop of the fit) simply discards the prefetched numerators.  Elsewhere: identical to
 * nmfb200_nmf_loss. */
int nmfb200_nmf_loss_prefetch_w(nmfb200_ctx* ctx, const float* W, const float* H, double beta,
                                double* loss_dev, void* stream);

/* Row-sharded W update (SURVEY.md 8e).  `partial` is a device fp32 buffer of
 * nmfb200_nmf_w_partial_numel() elements receiving this shard's raw numerator (C*R), then either
 * colsum(H_local) (R, beta == 1) or the raw denominator (C*R).  The caller sum-all-reduces it and
 * passes the reduced buffer to _w_apply, which performs nmf.py:78-92 on every rank identically. */
int64_t nmfb200_nmf_w_partial_numel(const nmfb200_ctx* ctx, double beta);
int nmfb200_nmf_w_partial(nmfb200_ctx* ctx, const float* W, const float* H, double beta,
                          float* partial, void* stream);
/* Raw terms of the multiplicative update of ONE factor (which = 0: W, 1: H), computed from the current W and H without
 * touching either: `out` receives the numerator relu-free (rows*R: the first backward pass of nmf.py:76-78 /
 * trainer.py:91-93), then colsum(other factor) (R, beta == 1: nmf.py:122-131) or the raw denominator (rows*R: the second
 * backward pass, nmf.py:82 / trainer.py:95-96).  This is what torchnmf.trainer.BetaMu.step (trainer.py:36-121) and
 * torchnmf.plca (plca.py:252-253: the simultaneous W / H / Z updates from ONE V / (W Z H) ratio) are built from. */
int64_t nmfb200_nmf_raw_terms_numel(const nmfb200_ctx* ctx, int which, double beta);
int nmfb200_nmf_raw_terms(nmfb200_ctx* ctx, const float* W, const float* H, int which, double beta,
                          float* out, void* stream);
int nmfb200_nmf_w_apply(nmfb200_ctx* ctx, float* W, const float* reduced,
                        double beta, double gamma, double l1_reg, double l2_reg, void* stream);

/* Sparse target for beta 1 and beta 2 (nmf.py:603-638 `_nmf_sp_recon_beta_pos_neg`, :95-119): registers V (N x C) in both
 * compressed forms -- CSR (crow[N+1], col[nnz], val[nnz]) and CSC = CSR of V^T (ccol[C+1], row[nnz], val_t[nnz]) -- int64
 * indices, fp32 values, device pointers borrowed until the next set_target*.  v_norm_kl / v_norm_eu: `_get_V_norm` nmf.py:161-170
 * for beta 1 / 2.  update_w / update_h / iterate / loss then evaluate the update terms at the non-zeros only (one warp per row
 * or column, fp32) and never form the dense product; any other beta returns NMFB200_ERR_INVALID (densify the target). */
int nmfb200_nmf_set_target_sparse(nmfb200_ctx* ctx, int64_t nnz, const int64_t* crow, const int64_t* col, const float* val,
                                  const int64_t* ccol, const int64_t* row, const float* val_t,
                                  double v_norm_kl, double v_norm_eu, void* stream);

/* Row-sharded W update over PEER MEMORY (ranks of one NVLink domain, one process per GPU, 2..8 ranks) -- the fused form of
 * w_partial -> all-reduce -> w_apply above, without a collective library call on the data path:
 *   local contraction -> a pack kernel that pushes this rank's partial [C*R | R] into its slot of EVERY rank's exchange block
 *   (posted NVLink writes) and publishes its iteration counter -> ONE ratio-stage kernel per rank that waits for all counters,
 *   sums the slots of its own block in rank order (the replicas of W stay bit-identical) and applies nmf.py:78-92.
 * Setup (once per context, collective): peer_alloc returns this rank's 64-byte CUDA IPC handle; exchange the handles (any
 * transport; the Python host side uses torch.distributed); peer_connect takes all `world` handles in rank order.  Then every
 * rank calls update_w_peer for every W update.  peer_supported: 1 if this context / beta can use it (tensor-core path,
 * rank % 4 == 0, beta != 2).  A rank that never arrives makes the kernel give up after ~2 s; nmfb200_ctx_check_health reports it. */
int nmfb200_nmf_peer_supported(const nmfb200_ctx* ctx, double beta);
int nmfb200_nmf_peer_alloc(nmfb200_ctx* ctx, void* ipc_handle_out /* 64 bytes */);
int nmfb200_nmf_peer_connect(nmfb200_ctx* ctx, int world, int rank, const void* ipc_handles /* world x 64 bytes */);
int nmfb200_nmf_peer_world(const nmfb200_ctx* ctx);          /* connected ranks, 0 if none */
int nmfb200_nmf_peer_release(nmfb200_ctx* ctx);
int nmfb200_nmf_update_w_peer(nmfb200_ctx* ctx, float* W, const float* H,
                              double beta, double gamma, double l1_reg, double l2_reg, void* stream);

/* Profiling aid for bench.py's roofline line: launches ONLY the fused contraction kernel of the W update
 * (which = 0) or the H update (which = 1) into the engine's scratch, leaving W and H untouched. */
int nmfb200_nmf_contract_only(nmfb200_ctx* ctx, const float* W, const float* H, int which, double beta,
                              void* stream);

/* ---- NMFD (1-D convolutive NMF) ---------------------------------------------------------- */

/* Sizes as NMFD.__init__ (nmf.py:762-774): V (B,C,L), W (C,R,T), H (B,R,L-T+1). */
int nmfb200_nmfd_create(nmfb200_ctx** out, int device, int64_t B, int64_t C, int64_t L,
                        int64_t R, int64_t T, int precision);
/* NMF2D / NMF3D (nmf.py:782-865, :868-942: conv2d / conv3d with flipped kernels and full padding): the same context type
 * with ndim = 2 or 3 convolved axes.  vdims = the target's sizes over those axes, kdims = kernel_size; V (B,C,*vdims),
 * W (C,R,*kdims), H (B,R,*(vdims - kdims + 1)), all contiguous.  ndim = 1 is nmfb200_nmfd_create.  Every nmfb200_nmfd_*
 * call below serves these contexts; they run on the fp32 kernels (precision auto or f32). */
int nmfb200_nmfnd_create(nmfb200_ctx** out, int device, int64_t B, int64_t C, int ndim, const int64_t* vdims,
                         int64_t R, const int64_t* kdims, int precision);
int nmfb200_nmfd_set_target(nmfb200_ctx* ctx, const float* V, void* stream);
int nmfb200_nmfd_update_w(nmfb200_ctx* ctx, float* W, const float* H,
                          double beta, double gamma, double l1_reg, double l2_reg, void* stream);
int nmfb200_nmfd_update_h(nmfb200_ctx* ctx, const float* W, float* H,
                          double beta, double gamma, double l1_reg, double l2_reg, void* stream);
int nmfb200_nmfd_loss(nmfb200_ctx* ctx, const float* W, const float* H, double beta,
                      double* loss_dev, void* stream);
/* The convolutive counterpart of nmfb200_nmf_raw_terms: both backward passes of ONE factor (which = 0: W, 1: H) through
 * the conv1d / conv2d / conv3d reconstruction (nmf.py:776-779, :862-865, :938-942) from the current W and H, neither
 * touched.  `out` = raw numerator (the factor's numel), then colsum(other factor) (R, beta == 1) or the raw denominator
 * (numel).  With W := W * Z this is one EM step's gradients of torchnmf.plca.SIPLCA / SIPLCA2 / SIPLCA3
 * (plca.py:252-253 with the reconstructions :453-455, :534-537, :621-625), and BetaMu.step for the convolutive modules. */
int64_t nmfb200_nmfd_raw_terms_numel(const nmfb200_ctx* ctx, int which, double beta);
int nmfb200_nmfd_raw_terms(nmfb200_ctx* ctx, const float* W, const float* H, int which, double beta,
                           float* out, void* stream);
/* The caller changed W and / or H in place since the last call (the library keeps fp16 operand copies on the tensor-core
 * path and refreshes only what it knows changed): refresh both at the next call. */
int nmfb200_nmfd_sync_factors(nmfb200_ctx* ctx);

/* ---- sparseness-constrained NMF (Hoyer 2004) --------------------------------------------- */

/* Replaces torchnmf.nmf._proj_func (nmf.py:21-49) and the Python loops that call it once per component
 * (sparse_fit nmf.py:462-465, :472-475, :519-522, :565-568; trainer.SparsityProj.step trainer.py:176-181): every slice
 * x[:, j, :] of the fp32 device tensor x viewed as (outer, D, inner) is replaced IN PLACE by the closest non-negative
 * vector with L1 norm k1[j] and squared L2 norm k2[j] (k1, k2: D device floats).  The reference's data-dependent loop
 * (one host synchronisation per round and slice) runs on the device, one block per slice, one launch for all D slices.
 * zeroed_ws: D * outer * inner bytes of device scratch.  Context-free: runs on CUDA device `device`, the caller's
 * current device is restored. */
int nmfb200_hoyer_project(int device, float* x, int64_t outer, int64_t D, int64_t inner, const float* k1, const float* k2,
                          void* zeroed_ws, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NMF_B200_H_ */
