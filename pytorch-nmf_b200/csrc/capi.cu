// C ABI of libnmf_b200 (see include/nmf_b200.h): context management and the per-update call graphs.
#include "../../include/nmf_b200.h"

#include <atomic>
#include <new>

#include "common.cuh"
#include "tc_nmf.cuh"
#include "tc_nmfd.cuh"

namespace nmfb200 {
static thread_local std::string g_err;
static std::atomic<int64_t> g_launches{0};
void set_error(const std::string& msg) { g_err = msg; }
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
}  // namespace nmfb200

using namespace nmfb200;

struct nmfb200_ctx {
  int kind = 0;            // 0 = NMF, 1 = NMFD
  int device = 0;
  int precision = NMFB200_PREC_F32;
  bool auto_mode = false;   // precision AUTO: the tensor-core path is used only where it is known to hold the parity bar
  bool tc_off = false;      // AUTO found the target outside the fp16 operand range: fp32 CUDA-core kernels instead
  int64_t N = 0, C = 0, R = 0;
  NmfdShape d{};
  const float* V = nullptr;
  int64_t ldv = 0;
  bool has_target = false;
  // chunked partial numerators / denominators of the CUDA-core path
  float* num = nullptr;
  float* den = nullptr;
  int64_t part_floats = 0;
  int nch_w = 1, nch_h = 1;
  float* colsum = nullptr;        // [2][R]: 0 = colsum(W), 1 = colsum(H)
  float* cs_scratch = nullptr;
  int64_t cs_scratch_floats = 0;
  double* loss_blocks = nullptr;
  int loss_max_blocks = 0;
  float* mm_scratch = nullptr;    // 2048 + 2
  // sparse target (beta 1 / 2): borrowed CSR (rows of V) and CSC (= CSR of V^T) forms, V_norm of nmf.py:161-170
  bool sparse = false;
  const int64_t *sp_crow = nullptr, *sp_col = nullptr, *sp_ccol = nullptr, *sp_row = nullptr;
  const float *sp_val = nullptr, *sp_val_t = nullptr;
  double sp_vnorm_kl = 0.0, sp_vnorm_eu = 0.0;
  float* sp_gram = nullptr;       // [2][R*R] (W^T W, H^T H) + per-block partials
  double* sp_loss_part = nullptr;
  // NMFD
  float* Pn = nullptr;
  float* Pp = nullptr;
  int wgrad_nsplit = 1;
  int dgrad_nsplit = 1;
  // tensor-core path state (tc_nmf.cu / tc_nmfd.cu)
  TcState* tc = nullptr;
  TcNmfdState* tcd = nullptr;
};

namespace {

int fail(int code, const std::string& msg) { set_error(msg); return code; }

// Every entry point runs on the context's device and leaves the calling thread's current device as it found it
// (a fit() on a module living on cuda:1 must not redirect the caller's later "cuda" allocations).
struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    int cur = -1;
    if (cudaGetDevice(&cur) != cudaSuccess) { ok = false; return; }
    if (cur != dev) {
      if (cudaSetDevice(dev) != cudaSuccess) { ok = false; return; }
      prev = cur;
    }
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;
};

#define CTX_GUARD(ctx, want_kind)                                                   \
  if (!(ctx)) return fail(NMFB200_ERR_INVALID, "null context");                     \
  if ((ctx)->kind != (want_kind)) return fail(NMFB200_ERR_INVALID, "wrong context kind"); \
  DeviceGuard _dev_guard((ctx)->device);                                            \
  if (!_dev_guard.ok) return fail(NMFB200_ERR_CUDA, "cannot select the context's device");

int chunks_for(int64_t rows, int64_t cols) {
  int64_t rb = ceil_div(rows, 64), tiles = ceil_div(cols, 64);
  int64_t want = ceil_div(148 * 4, rb);
  if (want > tiles) want = tiles;
  if (want > 32) want = 32;
  if (want < 1) want = 1;
  return (int)want;
}

int ensure_den(nmfb200_ctx* c) {
  if (!c->den) NMF_CUDA_CHECK(cudaMalloc(&c->den, c->part_floats * sizeof(float)));
  return 0;
}

void free_ctx(nmfb200_ctx* c) {
  if (!c) return;
  DeviceGuard guard(c->device);
  if (c->tc) tc_destroy(c->tc);
  if (c->tcd) tc_nmfd_destroy(c->tcd);
  cudaFree(c->num); cudaFree(c->den); cudaFree(c->colsum); cudaFree(c->cs_scratch);
  cudaFree(c->loss_blocks); cudaFree(c->mm_scratch); cudaFree(c->Pn); cudaFree(c->Pp);
  cudaFree(c->sp_gram); cudaFree(c->sp_loss_part);
  delete c;
}

// CUDA-core contraction of one NMF factor update (which = 0: W, 1: H) into c->num / c->den (chunked partials).
int simt_contract(nmfb200_ctx* c, int which, const float* W, const float* H, double beta, cudaStream_t st) {
  if (beta != 1.0) { int e = ensure_den(c); if (e) return e; }
  // W update: F = W (C rows), G = H (N rows), Vm = V^T;  H update: F = H, G = W, Vm = V
  const int64_t rows = which == 0 ? c->C : c->N;
  return simt_nmf_contract(c->V, c->ldv, /*trans=*/which == 0 ? 1 : 0, which == 0 ? W : H, which == 0 ? H : W, rows,
                           which == 0 ? c->N : c->C, (int)c->R, beta, which == 0 ? c->nch_w : c->nch_h, c->num, c->den,
                           c->R, rows * c->R, st);
}

bool use_tc(const nmfb200_ctx* c, double beta) {
  return c->tc != nullptr && !c->tc_off && tc_supports_beta(c->tc, beta);
}

// NMFD: beta = 1 on tensor cores (tc_nmfd.cu), everything else on the fp32 sliding GEMMs (nmfd.cu)
bool nmfd_use_tc(const nmfb200_ctx* c, double beta) { return c->tcd && !c->tc_off && beta == 1.0; }

}  // namespace

extern "C" {

int nmfb200_abi_version(void) { return NMFB200_ABI_VERSION; }
#ifndef NMFB200_SRC_HASH
#define NMFB200_SRC_HASH "unstamped"
#endif
#define NMFB200_STR2(x) #x
#define NMFB200_STR(x) NMFB200_STR2(x)
const char* nmfb200_build_info(void) {
  return "src=" NMFB200_SRC_HASH " nvcc=" NMFB200_STR(__CUDACC_VER_MAJOR__) "." NMFB200_STR(__CUDACC_VER_MINOR__) "."
         NMFB200_STR(__CUDACC_VER_BUILD__) " arch=sm_100a built=" __DATE__ " " __TIME__;
}
const char* nmfb200_last_error(void) { return g_err.c_str(); }
int64_t nmfb200_launch_count(void) { return g_launches.load(); }

int nmfb200_ctx_check_health(nmfb200_ctx* ctx, void* stream) {
  if (!ctx) return fail(NMFB200_ERR_INVALID, "null context");
  DeviceGuard guard(ctx->device);
  if (!guard.ok) return fail(NMFB200_ERR_CUDA, "cannot select the context's device");
  if (ctx->tc) {
    const int pr = tc_peer_check(ctx->tc, (cudaStream_t)stream);
    if (pr > 0) return fail(NMFB200_ERR_STATE, "a sharded W update gave up waiting for rank " + std::to_string(pr - 1) +
                                               "'s buffer; results are invalid");
    if (pr < 0) return fail(NMFB200_ERR_CUDA, "stream synchronize failed");
  }
  return nmfb200_check_health(stream);
}

int nmfb200_check_health(void* stream) {
  int rc = tc_check_wait_abort((cudaStream_t)stream);
  if (rc == 0) rc = tc_nmfd_check_wait_abort();
  if (rc > 0) return fail(NMFB200_ERR_STATE, "a kernel aborted an internal barrier wait; results are invalid");
  if (rc < 0) return fail(NMFB200_ERR_CUDA, std::string("stream synchronize: ") + cudaGetErrorString(cudaGetLastError()));
  return 0;
}

int nmfb200_nmf_create(nmfb200_ctx** out, int device, int64_t N, int64_t C, int64_t R, int precision) {
  if (!out) return fail(NMFB200_ERR_INVALID, "out is null");
  *out = nullptr;
  if (N < 1 || C < 1 || R < 1) return fail(NMFB200_ERR_INVALID, "N, C, R must be positive");
  if (R > 256) return fail(NMFB200_ERR_INVALID, "rank > 256 is not supported");
  if (precision < NMFB200_PREC_AUTO || precision > NMFB200_PREC_F16_SPLIT)
    return fail(NMFB200_ERR_INVALID, "unknown precision mode");
  DeviceGuard guard(device);
  if (!guard.ok) return fail(NMFB200_ERR_CUDA, "cannot select the requested device");
  nmfb200_ctx* c = new (std::nothrow) nmfb200_ctx();
  if (!c) return fail(NMFB200_ERR_INVALID, "out of host memory");
  c->kind = 0; c->device = device; c->N = N; c->C = C; c->R = R;
  int resolved = precision;
  // AUTO: single-rounded fp16 operands already hold the north-star parity with a 6x margin once the ratio tile is
  // kappa-centred (cfg2, 200 iterations vs the reference: max rel. error 1.7e-4 f16, 9.7e-5 f16_split; DESIGN.md 4.2)
  if (precision == NMFB200_PREC_AUTO) resolved = tc_shape_supported(N, C, R) ? NMFB200_PREC_F16 : NMFB200_PREC_F32;
  if (resolved != NMFB200_PREC_F32 && !tc_shape_supported(N, C, R)) {
    delete c;
    return fail(NMFB200_ERR_INVALID, "shape not supported by the tensor-core path (need R <= 128)");
  }
  c->precision = resolved;
  c->auto_mode = precision == NMFB200_PREC_AUTO;
  c->nch_w = chunks_for(C, N);
  c->nch_h = chunks_for(N, C);
  int64_t pf = (int64_t)c->nch_w * C * R;
  if ((int64_t)c->nch_h * N * R > pf) pf = (int64_t)c->nch_h * N * R;
  c->part_floats = pf;
  int64_t csf = colsum_scratch_floats(N > C ? N : C, (int)R, 1);
  c->cs_scratch_floats = csf;
  c->loss_max_blocks = simt_nmf_max_blocks(N, C);
  cudaError_t e = cudaSuccess;
  if (e == cudaSuccess) e = cudaMalloc(&c->num, pf * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&c->colsum, 2 * R * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&c->cs_scratch, csf * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&c->loss_blocks, (size_t)c->loss_max_blocks * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&c->mm_scratch, 2050 * sizeof(float));
  if (e != cudaSuccess) {
    free_ctx(c);
    return fail(NMFB200_ERR_CUDA, std::string("cudaMalloc: ") + cudaGetErrorString(e));
  }
  if (resolved != NMFB200_PREC_F32) {
    int rc = tc_create(&c->tc, device, N, C, R, resolved == NMFB200_PREC_F16_SPLIT);
    if (rc) { free_ctx(c); return rc; }
  }
  *out = c;
  return 0;
}

void nmfb200_destroy(nmfb200_ctx* ctx) { free_ctx(ctx); }

int nmfb200_precision(const nmfb200_ctx* ctx) {
  if (!ctx) return -100;
  return ctx->tc_off ? NMFB200_PREC_F32 : ctx->precision;
}

int nmfb200_precision_for_beta(const nmfb200_ctx* ctx, double beta) {
  if (!ctx) return -100;
  if (ctx->kind == 1) return nmfd_use_tc(ctx, beta) ? NMFB200_PREC_F16 : NMFB200_PREC_F32;
  if (ctx->kind != 0 || !use_tc(ctx, beta)) return NMFB200_PREC_F32;
  // beta != 1 kernels read only the hi halves of the operand copies
  return (beta == 1.0 || beta == 2.0) ? ctx->precision : NMFB200_PREC_F16;
}

int nmfb200_nmf_set_target(nmfb200_ctx* ctx, const float* V, int64_t ldv, void* stream) {
  CTX_GUARD(ctx, 0);
  if (!V || ldv < ctx->C) return fail(NMFB200_ERR_INVALID, "bad target pointer / leading dimension");
  cudaStream_t st = (cudaStream_t)stream;
  ctx->V = V; ctx->ldv = ldv; ctx->has_target = true; ctx->sparse = false;
  int rc = matrix_minmax(V, ctx->N, ctx->C, ldv, ctx->mm_scratch, ctx->mm_scratch + 2048, st);
  if (rc) return rc;
  ctx->tc_off = false;
  if (ctx->tc) {
    rc = tc_set_target(ctx->tc, V, ldv, ctx->mm_scratch + 2048, st);
    if (rc) return rc;
    if (ctx->auto_mode) {
      // AUTO is conservative: the fp16 copy of V carries ONE power-of-two scale (max -> 2^14), so positive entries below
      // max * 2^-28 lose precision or vanish (power spectrograms span more than that).  Targets with more than a
      // negligible share of such entries run on the fp32 kernels; asking for "f16" / "f16_split" explicitly keeps the
      // tensor cores.
      unsigned long long lossy = 0;
      rc = tc_target_lossy(ctx->tc, &lossy, st);
      if (rc) return rc;
      // a handful of tiny entries in a 10^8-cell matrix carry no structure; a quiet row / band (>= 1e-6 of the cells) does
      ctx->tc_off = (double)lossy > 1e-6 * (double)ctx->N * (double)ctx->C;
      // ... and for heavy-tailed targets (max / mean > 64: spectrogram-like, lognormal, ...).  Measured on the lognormal
      // fixtures of tests/golden/reference_r2.npz (30 iterations, tolerance rtol 1e-3): f16 34x, f16_split 2x, f32 0.1x of
      // the tolerance -- MU on such targets converges slowly and keeps the per-update operand rounding instead of
      // averaging it out as it does on well-conditioned data (uniform-like targets: 0.17x after 200 iterations).
      if (!ctx->tc_off) {
        double vsum = 0.0;
        float mm[2] = {0.f, 0.f};
        rc = tc_target_sum(ctx->tc, &vsum, st);
        if (rc) return rc;
        NMF_CUDA_CHECK(cudaMemcpyAsync(mm, ctx->mm_scratch + 2048, sizeof(mm), cudaMemcpyDeviceToHost, st));
        NMF_CUDA_CHECK(cudaStreamSynchronize(st));
        const double mean = vsum / ((double)ctx->N * (double)ctx->C);
        ctx->tc_off = !(mean > 0.0) || (double)mm[1] > 64.0 * mean;
      }
    }
  }
  return 0;
}

/* ---- sparse targets (beta 1 and 2): nmf.py:603-638 without the dense product ------------------------------ */

int nmfb200_nmf_set_target_sparse(nmfb200_ctx* ctx, int64_t nnz, const int64_t* crow, const int64_t* col, const float* val,
                                  const int64_t* ccol, const int64_t* row, const float* val_t, double v_norm_kl,
                                  double v_norm_eu, void* stream) {
  CTX_GUARD(ctx, 0);
  (void)stream;
  if (nnz < 0 || !crow || !ccol || (nnz > 0 && (!col || !val || !row || !val_t)))
    return fail(NMFB200_ERR_INVALID, "bad compressed sparse target");
  if (!ctx->sp_gram) {
    const int64_t R = ctx->R;
    NMF_CUDA_CHECK(cudaMalloc(&ctx->sp_gram, (size_t)(2 * R * R + sparse_gram_part_floats((int)R)) * sizeof(float)));
    NMF_CUDA_CHECK(cudaMalloc(&ctx->sp_loss_part, (size_t)sparse_loss_blocks(ctx->N) * sizeof(double)));
  }
  ctx->sp_crow = crow; ctx->sp_col = col; ctx->sp_val = val; ctx->sp_ccol = ccol; ctx->sp_row = row; ctx->sp_val_t = val_t;
  ctx->sp_vnorm_kl = v_norm_kl; ctx->sp_vnorm_eu = v_norm_eu;
  ctx->sparse = true; ctx->has_target = true; ctx->V = nullptr; ctx->tc_off = true;      // the dense kernels are out of play
  return 0;
}

namespace {
// The ratio stage's input for one dense-NMF factor (which = 0: W, 1: H; rows x R, row pitch R): `nchunks` slabs of partial
// numerators (and denominators, beta != 1) or, for beta 1, the column sum `kl` of the other factor as the denominator.
ApplyArgs nmf_apply_args(const nmfb200_ctx* ctx, int which, const float* num, const float* den, const float* kl,
                         int nchunks) {
  ApplyArgs a{};
  a.numel = (which == 0 ? ctx->C : ctx->N) * ctx->R; a.R = (int)ctx->R; a.inner = 1; a.rowlen = ctx->R; a.ldp = ctx->R;
  a.num = num; a.den = den; a.kl_den = kl; a.nchunks = nchunks; a.chunk_stride = a.numel;
  return a;
}

// Both terms of one dense-NMF factor update (which = 0: W, 1: H) from the current factors, described as the ratio stage's
// input.  Dense target: the CUDA-core contraction's chunked partials.  Sparse target: the numerator at the non-zeros of the
// compressed form whose segments are that factor's rows (W over CSC, H over CSR), and for beta 2 the denominator as the
// factor's rows times the Gram matrix of the other factor (nmf.py:609).  Beta 1 divides by the column sum of the other
// factor (nmf.py:122-131).  Shared by the update and by nmfb200_nmf_raw_terms; the tensor-core path has its own fused
// ratio stage.
int nmf_terms(nmfb200_ctx* ctx, const float* W, const float* H, int which, double beta, ApplyArgs& a, cudaStream_t st) {
  const int R = (int)ctx->R;
  const int64_t rows = which == 0 ? ctx->C : ctx->N, orows = which == 0 ? ctx->N : ctx->C;
  const float* other = which == 0 ? H : W;
  int rc, nchunks = 1;
  if (ctx->sparse) {
    if (beta != 1.0 && beta != 2.0) return fail(NMFB200_ERR_INVALID, "sparse targets: beta must be 1 or 2 (densify the target for other beta)");
    const int64_t* ptr = which == 0 ? ctx->sp_ccol : ctx->sp_crow;
    const int64_t* idx = which == 0 ? ctx->sp_row : ctx->sp_col;
    const float* val = which == 0 ? ctx->sp_val_t : ctx->sp_val;
    const float* F = which == 0 ? W : H;
    rc = sparse_numerator(ptr, idx, val, F, other, R, rows, beta, ctx->num, st);
    if (rc == 0 && beta == 2.0) {
      rc = ensure_den(ctx);
      if (rc) return rc;
      float* G = ctx->sp_gram + (1 - which) * R * R;
      rc = sparse_gram(other, orows, R, ctx->sp_gram + 2 * R * R, G, st);
      if (rc == 0) rc = sparse_rows_times_gram(F, G, rows, R, ctx->den, st);
    }
  } else {
    nchunks = which == 0 ? ctx->nch_w : ctx->nch_h;
    rc = simt_contract(ctx, which, W, H, beta, st);
  }
  if (rc) return rc;
  float* kl = nullptr;
  if (beta == 1.0) {
    kl = ctx->colsum + (1 - which) * R;
    rc = factor_colsum(other, orows, R, 1, ctx->cs_scratch, ctx->cs_scratch_floats, kl, st);
    if (rc) return rc;
  }
  a = nmf_apply_args(ctx, which, ctx->num, beta == 1.0 ? nullptr : ctx->den, kl, nchunks);
  return 0;
}

// nmf.py:78-92 on the terms `a` of one factor; the tensor-core operand copy of that factor is stale afterwards.
int nmf_apply(nmfb200_ctx* ctx, int which, ApplyArgs a, float* param, double gamma, double l1_reg, double l2_reg,
              cudaStream_t st) {
  a.param = param; a.gamma = (float)gamma; a.l1 = (float)l1_reg; a.l2 = (float)l2_reg;
  int rc = apply_update(a, st);
  if (rc) return rc;
  if (ctx->tc) tc_mark_dirty(ctx->tc, which == 0, which == 1);
  return 0;
}

int nmf_update(nmfb200_ctx* ctx, const float* W, const float* H, int which, float* param, double beta, double gamma,
               double l1_reg, double l2_reg, cudaStream_t st) {
  if (use_tc(ctx, beta))
    return which == 0 ? tc_update_w(ctx->tc, param, H, beta, gamma, l1_reg, l2_reg, st)
                      : tc_update_h(ctx->tc, W, param, beta, gamma, l1_reg, l2_reg, st);
  ApplyArgs a;
  int rc = nmf_terms(ctx, W, H, which, beta, a, st);
  if (rc) return rc;
  return nmf_apply(ctx, which, a, param, gamma, l1_reg, l2_reg, st);
}

// nmfb200_nmf_raw_terms past its argument checks: [numerator rows x R | colsum(other) R (beta 1) or denominator rows x R]
int nmf_raw_terms(nmfb200_ctx* ctx, const float* W, const float* H, int which, double beta, float* out, cudaStream_t st) {
  if (use_tc(ctx, beta) && tc_supports_partial(ctx->tc, beta)) return tc_raw_terms(ctx->tc, which, W, H, beta, out, st);
  ApplyArgs a;
  int rc = nmf_terms(ctx, W, H, which, beta, a, st);
  if (rc) return rc;
  rc = raw_sum(a, out, out + a.numel, st);
  if (rc) return rc;
  if (beta == 1.0)
    NMF_CUDA_CHECK(cudaMemcpyAsync(out + a.numel, a.kl_den, (size_t)ctx->R * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return 0;
}

int sparse_loss_ctx(nmfb200_ctx* ctx, const float* W, const float* H, double beta, double* loss_dev, cudaStream_t st) {
  if (beta != 1.0 && beta != 2.0) return fail(NMFB200_ERR_INVALID, "sparse targets: beta must be 1 or 2");
  const int R = (int)ctx->R;
  const float *pa, *pb;
  int rc;
  if (beta == 1.0) {
    rc = factor_colsum(W, ctx->C, R, 1, ctx->cs_scratch, ctx->cs_scratch_floats, ctx->colsum, st);
    if (rc == 0) rc = factor_colsum(H, ctx->N, R, 1, ctx->cs_scratch, ctx->cs_scratch_floats, ctx->colsum + R, st);
    pa = ctx->colsum; pb = ctx->colsum + R;
  } else {
    rc = sparse_gram(W, ctx->C, R, ctx->sp_gram + 2 * R * R, ctx->sp_gram, st);
    if (rc == 0) rc = sparse_gram(H, ctx->N, R, ctx->sp_gram + 2 * R * R, ctx->sp_gram + R * R, st);
    pa = ctx->sp_gram; pb = ctx->sp_gram + R * R;
  }
  if (rc) return rc;
  return sparse_loss(ctx->sp_crow, ctx->sp_col, ctx->sp_val, H, W, R, ctx->N, beta, pa, pb,
                     beta == 1.0 ? ctx->sp_vnorm_kl : ctx->sp_vnorm_eu, ctx->sp_loss_part, loss_dev, st);
}
}  // namespace

int nmfb200_target_minmax(nmfb200_ctx* ctx, float* vmin, float* vmax, void* stream) {
  if (!ctx) return fail(NMFB200_ERR_INVALID, "null context");
  DeviceGuard guard(ctx->device);
  if (!guard.ok) return fail(NMFB200_ERR_CUDA, "cannot select the context's device");
  if (!ctx->has_target) return fail(NMFB200_ERR_STATE, "set_target has not been called");
  float mm[2];
  NMF_CUDA_CHECK(cudaMemcpyAsync(mm, ctx->mm_scratch + 2048, sizeof(mm), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  NMF_CUDA_CHECK(cudaStreamSynchronize((cudaStream_t)stream));
  if (vmin) *vmin = mm[0];
  if (vmax) *vmax = mm[1];
  return 0;
}

int nmfb200_nmf_sync_factors(nmfb200_ctx* ctx, const float* W, const float* H, void* stream) {
  CTX_GUARD(ctx, 0);
  if (!W || !H) return fail(NMFB200_ERR_INVALID, "null factor pointer");
  if (ctx->tc) tc_mark_dirty(ctx->tc, true, true);
  return 0;   // operand copies are rebuilt lazily; the CUDA-core path reads the fp32 factors directly
}

int nmfb200_nmf_update_w(nmfb200_ctx* ctx, float* W, const float* H, double beta, double gamma, double l1_reg,
                         double l2_reg, void* stream) {
  CTX_GUARD(ctx, 0);
  if (!ctx->has_target) return fail(NMFB200_ERR_STATE, "set_target has not been called");
  if (!W || !H) return fail(NMFB200_ERR_INVALID, "null factor pointer");
  return nmf_update(ctx, W, H, 0, W, beta, gamma, l1_reg, l2_reg, (cudaStream_t)stream);
}

int nmfb200_nmf_update_h(nmfb200_ctx* ctx, const float* W, float* H, double beta, double gamma, double l1_reg,
                         double l2_reg, void* stream) {
  CTX_GUARD(ctx, 0);
  if (!ctx->has_target) return fail(NMFB200_ERR_STATE, "set_target has not been called");
  if (!W || !H) return fail(NMFB200_ERR_INVALID, "null factor pointer");
  return nmf_update(ctx, W, H, 1, H, beta, gamma, l1_reg, l2_reg, (cudaStream_t)stream);
}

int nmfb200_nmf_iterate(nmfb200_ctx* ctx, float* W, float* H, double beta, double gamma, double l1_reg,
                        double l2_reg, int n_iter, void* stream) {
  CTX_GUARD(ctx, 0);
  if (!ctx->has_target) return fail(NMFB200_ERR_STATE, "set_target has not been called");
  if (!W || !H || n_iter < 0) return fail(NMFB200_ERR_INVALID, "bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  if (use_tc(ctx, beta)) return tc_iterate(ctx->tc, W, H, beta, gamma, l1_reg, l2_reg, n_iter, st);
  for (int i = 0; i < n_iter; ++i) {
    int rc = nmf_update(ctx, W, H, 0, W, beta, gamma, l1_reg, l2_reg, st);
    if (rc == 0) rc = nmf_update(ctx, W, H, 1, H, beta, gamma, l1_reg, l2_reg, st);
    if (rc) return rc;
  }
  return 0;
}

int nmfb200_nmf_loss(nmfb200_ctx* ctx, const float* W, const float* H, double beta, double* loss_dev,
                     void* stream) {
  CTX_GUARD(ctx, 0);
  if (!ctx->has_target) return fail(NMFB200_ERR_STATE, "set_target has not been called");
  if (!W || !H || !loss_dev) return fail(NMFB200_ERR_INVALID, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (ctx->sparse) return sparse_loss_ctx(ctx, W, H, beta, loss_dev, st);
  if (use_tc(ctx, beta)) return tc_loss(ctx->tc, W, H, beta, loss_dev, st);
  return simt_nmf_loss(ctx->V, ctx->ldv, H, W, ctx->N, ctx->C, (int)ctx->R, beta, ctx->loss_blocks,
                       ctx->loss_max_blocks, loss_dev, st);
}

int nmfb200_nmf_loss_prefetch_w(nmfb200_ctx* ctx, const float* W, const float* H, double beta, double* loss_dev,
                                void* stream) {
  CTX_GUARD(ctx, 0);
  if (!ctx->has_target) return fail(NMFB200_ERR_STATE, "set_target has not been called");
  if (!W || !H || !loss_dev) return fail(NMFB200_ERR_INVALID, "null pointer");
  if (!ctx->sparse && use_tc(ctx, beta))
    return tc_loss_prefetch_w(ctx->tc, W, H, beta, loss_dev, (cudaStream_t)stream);
  return nmfb200_nmf_loss(ctx, W, H, beta, loss_dev, stream);
}

int64_t nmfb200_nmf_raw_terms_numel(const nmfb200_ctx* ctx, int which, double beta) {
  if (!ctx || ctx->kind != 0 || (which != 0 && which != 1)) return -1;
  const int64_t rows = which == 0 ? ctx->C : ctx->N;
  return beta == 1.0 ? rows * ctx->R + ctx->R : 2 * rows * ctx->R;
}

int nmfb200_nmf_raw_terms(nmfb200_ctx* ctx, const float* W, const float* H, int which, double beta, float* out,
                          void* stream) {
  CTX_GUARD(ctx, 0);
  if (!ctx->has_target) return fail(NMFB200_ERR_STATE, "set_target has not been called");
  if (ctx->sparse) return fail(NMFB200_ERR_STATE, "not available for a sparse target");
  if (!W || !H || !out || (which != 0 && which != 1)) return fail(NMFB200_ERR_INVALID, "bad argument");
  return nmf_raw_terms(ctx, W, H, which, beta, out, (cudaStream_t)stream);
}

// The sharded W update's partial is the W update's raw terms.
int64_t nmfb200_nmf_w_partial_numel(const nmfb200_ctx* ctx, double beta) { return nmfb200_nmf_raw_terms_numel(ctx, 0, beta); }

int nmfb200_nmf_w_partial(nmfb200_ctx* ctx, const float* W, const float* H, double beta, float* partial,
                          void* stream) {
  CTX_GUARD(ctx, 0);
  if (!ctx->has_target) return fail(NMFB200_ERR_STATE, "set_target has not been called");
  if (ctx->sparse) return fail(NMFB200_ERR_STATE, "not available for a sparse target");
  if (!W || !H || !partial) return fail(NMFB200_ERR_INVALID, "null pointer");
  return nmf_raw_terms(ctx, W, H, 0, beta, partial, (cudaStream_t)stream);
}

/* ---- row-sharded W update over peer memory (NVLink, one process per GPU) ---------------------- */

int nmfb200_nmf_peer_supported(const nmfb200_ctx* ctx, double beta) {
  if (!ctx || ctx->kind != 0 || !ctx->tc || ctx->tc_off || !ctx->has_target) return 0;
  return (tc_supports_beta(ctx->tc, beta) && tc_peer_supported(ctx->tc, beta)) ? 1 : 0;
}

int nmfb200_nmf_peer_alloc(nmfb200_ctx* ctx, void* ipc_handle_out) {
  CTX_GUARD(ctx, 0);
  if (!ctx->tc) return fail(NMFB200_ERR_STATE, "the peer-memory W update needs the tensor-core path");
  if (!ipc_handle_out) return fail(NMFB200_ERR_INVALID, "null pointer");
  return tc_peer_alloc(ctx->tc, ipc_handle_out);
}

int nmfb200_nmf_peer_connect(nmfb200_ctx* ctx, int world, int rank, const void* ipc_handles) {
  CTX_GUARD(ctx, 0);
  if (!ctx->tc) return fail(NMFB200_ERR_STATE, "the peer-memory W update needs the tensor-core path");
  if (!ipc_handles) return fail(NMFB200_ERR_INVALID, "null pointer");
  return tc_peer_connect(ctx->tc, world, rank, ipc_handles);
}

int nmfb200_nmf_peer_world(const nmfb200_ctx* ctx) {
  return (ctx && ctx->kind == 0 && ctx->tc) ? tc_peer_world(ctx->tc) : 0;
}

int nmfb200_nmf_peer_release(nmfb200_ctx* ctx) {
  CTX_GUARD(ctx, 0);
  if (ctx->tc) tc_peer_release(ctx->tc);
  return 0;
}

int nmfb200_nmf_update_w_peer(nmfb200_ctx* ctx, float* W, const float* H, double beta, double gamma, double l1_reg,
                              double l2_reg, void* stream) {
  CTX_GUARD(ctx, 0);
  if (!ctx->has_target) return fail(NMFB200_ERR_STATE, "set_target has not been called");
  if (!W || !H) return fail(NMFB200_ERR_INVALID, "null factor pointer");
  if (!nmfb200_nmf_peer_supported(ctx, beta)) return fail(NMFB200_ERR_STATE, "peer-memory W update is not available for this context / beta");
  return tc_update_w_peer(ctx->tc, W, H, beta, gamma, l1_reg, l2_reg, (cudaStream_t)stream);
}

int nmfb200_nmf_w_apply(nmfb200_ctx* ctx, float* W, const float* reduced, double beta, double gamma,
                        double l1_reg, double l2_reg, void* stream) {
  CTX_GUARD(ctx, 0);
  if (!W || !reduced) return fail(NMFB200_ERR_INVALID, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (use_tc(ctx, beta)) return tc_w_apply(ctx->tc, W, reduced, beta, gamma, l1_reg, l2_reg, st);
  const float* den = reduced + ctx->C * ctx->R;          // [numerator C x R | colsum(H) R (beta 1) or denominator C x R]
  const ApplyArgs a = nmf_apply_args(ctx, 0, reduced, beta == 1.0 ? nullptr : den, beta == 1.0 ? den : nullptr, 1);
  return nmf_apply(ctx, 0, a, W, gamma, l1_reg, l2_reg, st);
}

int nmfb200_nmf_contract_only(nmfb200_ctx* ctx, const float* W, const float* H, int which, double beta,
                              void* stream) {
  CTX_GUARD(ctx, 0);
  if (!ctx->has_target) return fail(NMFB200_ERR_STATE, "set_target has not been called");
  if (ctx->sparse) return fail(NMFB200_ERR_STATE, "not available for a sparse target");
  if (!W || !H) return fail(NMFB200_ERR_INVALID, "null factor pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (use_tc(ctx, beta)) return tc_contract_only(ctx->tc, W, H, which, beta, st);
  return simt_contract(ctx, which, W, H, beta, st);
}

/* ---- NMFD ------------------------------------------------------------------------------------ */

// One context type serves NMFD (one sliding axis) and NMF2D / NMF3D (the last axis slides, the outer ones are loops):
// vdims / kdims hold the target's and the kernel's sizes over the ndim convolved axes.
static int nmfd_create_impl(nmfb200_ctx** out, int device, int64_t B, int64_t C, int ndim, const int64_t* vdims,
                            int64_t R, const int64_t* kdims, int precision) {
  if (!out) return fail(NMFB200_ERR_INVALID, "out is null");
  *out = nullptr;
  if (ndim < 1 || ndim > 3 || !vdims || !kdims) return fail(NMFB200_ERR_INVALID, "1 to 3 convolved axes are supported");
  int64_t X[3] = {1, 1, 1}, K[3] = {1, 1, 1};            // right-aligned: X[2] / K[2] is the last (sliding) axis
  for (int i = 0; i < ndim; ++i) { X[3 - ndim + i] = vdims[i]; K[3 - ndim + i] = kdims[i]; }
  const int64_t L = X[2], T = K[2];
  if (B < 1 || C < 1 || R < 1) return fail(NMFB200_ERR_INVALID, "bad NMFD sizes");
  for (int i = 0; i < 3; ++i)
    if (K[i] < 1 || X[i] < K[i]) return fail(NMFB200_ERR_INVALID, "bad NMFD sizes");
  if (R > 256) return fail(NMFB200_ERR_INVALID, "rank > 256 is not supported");
  if (precision != NMFB200_PREC_AUTO && precision != NMFB200_PREC_F32 && precision != NMFB200_PREC_F16)
    return fail(NMFB200_ERR_INVALID, "NMFD precision must be auto, f32 or f16");
  if (B * C * X[0] * X[1] * L > (int64_t)1 << 40 || X[0] * X[1] * L > (int64_t)1 << 30 || K[0] * K[1] * T > (int64_t)1 << 24)
    return fail(NMFB200_ERR_INVALID, "NMFD target too large");
  const bool one_d = X[0] == 1 && X[1] == 1;
  if (!one_d && precision == NMFB200_PREC_F16)
    return fail(NMFB200_ERR_INVALID, "NMF2D / NMF3D run on the fp32 kernels (precision auto or f32)");
  NmfdShape d{(int)B, (int)C, (int)L, (int)R, (int)T, (int)(L - T + 1)};
  d.X1 = (int)X[0]; d.X2 = (int)X[1]; d.T1 = (int)K[0]; d.T2 = (int)K[1];
  // AUTO: the tensor-core kernels wherever they compute the shape (beta = 1 only: nmfd_use_tc); fp32 everywhere else
  const bool tc_shape = tc_nmfd_shape_supported(d);
  if (precision == NMFB200_PREC_F16 && !tc_shape)
    return fail(NMFB200_ERR_INVALID, "shape not supported by the tensor-core NMFD path (need T <= 128)");
  DeviceGuard guard(device);
  if (!guard.ok) return fail(NMFB200_ERR_CUDA, "cannot select the requested device");
  nmfb200_ctx* c = new (std::nothrow) nmfb200_ctx();
  if (!c) return fail(NMFB200_ERR_INVALID, "out of host memory");
  c->kind = 1; c->device = device; c->R = R;
  c->precision = (precision == NMFB200_PREC_F16 || (precision == NMFB200_PREC_AUTO && tc_shape)) ? NMFB200_PREC_F16 : NMFB200_PREC_F32;
  c->auto_mode = precision == NMFB200_PREC_AUTO;
  c->d = d;
  c->dgrad_nsplit = nmfd_dgrad_nsplit(c->d);
  c->wgrad_nsplit = nmfd_wgrad_nsplit(c->d);
  int64_t pf = (int64_t)c->wgrad_nsplit * C * R * c->d.w_inner();
  int64_t hf = (int64_t)c->dgrad_nsplit * B * R * c->d.h_inner();
  if (hf > pf) pf = hf;
  c->part_floats = pf;
  int64_t cs1 = colsum_scratch_floats(C, (int)R, c->d.w_inner()), cs2 = colsum_scratch_floats(B, (int)R, c->d.h_inner());
  c->cs_scratch_floats = cs1 > cs2 ? cs1 : cs2;
  c->loss_max_blocks = nmfd_max_blocks(c->d);
  cudaError_t e = cudaSuccess;
  if (e == cudaSuccess) e = cudaMalloc(&c->num, pf * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&c->colsum, 2 * R * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&c->cs_scratch, c->cs_scratch_floats * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&c->loss_blocks, (size_t)c->loss_max_blocks * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&c->mm_scratch, 2050 * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&c->Pn, (size_t)B * C * c->d.v_inner() * sizeof(float));
  if (e != cudaSuccess) {
    free_ctx(c);
    return fail(NMFB200_ERR_CUDA, std::string("cudaMalloc: ") + cudaGetErrorString(e));
  }
  if (c->precision == NMFB200_PREC_F16) {
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess && prop.major == 10) {
      int rc = tc_nmfd_create(&c->tcd, c->d);          // beta = 1 runs as tcgen05 sliding GEMMs (tc_nmfd.cu)
      if (rc) { free_ctx(c); return rc; }
    } else if (precision == NMFB200_PREC_F16) {
      free_ctx(c);
      return fail(NMFB200_ERR_INVALID, "the tensor-core NMFD path needs an sm_100 device");
    }
  }
  *out = c;
  return 0;
}

int nmfb200_nmfd_create(nmfb200_ctx** out, int device, int64_t B, int64_t C, int64_t L, int64_t R, int64_t T,
                        int precision) {
  return nmfd_create_impl(out, device, B, C, 1, &L, R, &T, precision);
}

int nmfb200_nmfnd_create(nmfb200_ctx** out, int device, int64_t B, int64_t C, int ndim, const int64_t* vdims,
                         int64_t R, const int64_t* kdims, int precision) {
  return nmfd_create_impl(out, device, B, C, ndim, vdims, R, kdims, precision);
}

int nmfb200_nmfd_set_target(nmfb200_ctx* ctx, const float* V, void* stream) {
  CTX_GUARD(ctx, 1);
  if (!V) return fail(NMFB200_ERR_INVALID, "null target");
  ctx->V = V; ctx->has_target = true;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t vin = ctx->d.v_inner();
  int rc = matrix_minmax(V, (int64_t)ctx->d.B * ctx->d.C, vin, vin, ctx->mm_scratch, ctx->mm_scratch + 2048, st);
  if (rc) return rc;
  ctx->tc_off = false;
  if (ctx->tcd) {
    double vsum = 0.0;
    rc = tc_nmfd_set_target(ctx->tcd, V, &vsum, st);       // synchronises: sum(V) for kappa
    if (rc) return rc;
    tc_nmfd_mark_dirty(ctx->tcd);                         // a new fit: the factors may be anything
    if (ctx->auto_mode) {                                 // same conservative rule as the NMF path: heavy-tailed targets stay fp32
      float mm[2] = {0.f, 0.f};
      NMF_CUDA_CHECK(cudaMemcpyAsync(mm, ctx->mm_scratch + 2048, sizeof(mm), cudaMemcpyDeviceToHost, st));
      NMF_CUDA_CHECK(cudaStreamSynchronize(st));
      const double mean = vsum / ((double)ctx->d.B * ctx->d.C * ctx->d.L);
      ctx->tc_off = !(mean > 0.0) || (double)mm[1] > 64.0 * mean;
    }
  }
  return 0;
}

static int nmfd_phi(nmfb200_ctx* c, const float* W, const float* H, double beta, cudaStream_t st) {
  if (beta != 1.0) {
    if (!c->Pp) NMF_CUDA_CHECK(cudaMalloc(&c->Pp, (size_t)c->d.B * c->d.C * c->d.v_inner() * sizeof(float)));
    int e = ensure_den(c);
    if (e) return e;
  }
  return nmfd_recon_phi(c->d, c->V, W, H, beta, c->Pn, c->Pp, nullptr, 0, nullptr, st);
}

// Both backward passes of one factor (which = 0: W, 1: H) from the current factors, described as the ratio stage's input:
// split partial numerators (+ denominators for beta != 1), the KL column sums, the centring term of the tensor-core path.
// Shared by the update (nmf.py:367-391) and by nmfb200_nmfd_raw_terms.  `tc` reports which path produced the terms.
static int nmfd_terms(nmfb200_ctx* ctx, const float* W, const float* H, int which, double beta, ApplyArgs& a, bool* tc,
                      cudaStream_t st) {
  const NmfdShape& d = ctx->d;
  const int64_t inner = which == 0 ? d.w_inner() : d.h_inner();
  a = ApplyArgs{};
  a.numel = (int64_t)(which == 0 ? d.C : d.B) * d.R * inner; a.R = d.R; a.inner = inner; a.rowlen = (int64_t)d.R * inner;
  a.chunk_stride = a.numel; a.ldp = a.rowlen; a.absmax_bits = nullptr;
  *tc = nmfd_use_tc(ctx, beta);
  if (*tc) {
    int rc = tc_nmfd_recon(ctx->tcd, ctx->V, W, H, false, nullptr, st);
    if (rc) return rc;
    const float* part; int nsplit;
    rc = which == 0 ? tc_nmfd_wgrad(ctx->tcd, &part, &nsplit, st) : tc_nmfd_dgrad(ctx->tcd, &part, &nsplit, st);
    if (rc) return rc;
    a.num = part; a.den = nullptr; a.nchunks = nsplit;
    const float* cs = tc_nmfd_colsum(ctx->tcd) + (which == 0 ? d.R : 0);       // [colsum_W | colsum_H]
    a.kl_den = cs; a.kappa = tc_nmfd_kappa(ctx->tcd); a.kappa_vec = cs;
    return 0;
  }
  if (ctx->tcd) tc_nmfd_mark_dirty(ctx->tcd);            // this pass bypasses the tensor-core state
  int rc = nmfd_phi(ctx, W, H, beta, st);
  if (rc) return rc;
  const int nsplit = which == 0 ? ctx->wgrad_nsplit : ctx->dgrad_nsplit;
  rc = which == 0 ? nmfd_wgrad(d, ctx->Pn, H, ctx->num, nsplit, st) : nmfd_dgrad(d, ctx->Pn, W, ctx->num, nsplit, st);
  if (rc) return rc;
  float* kl = nullptr;
  if (beta == 1.0) {                                     // nmf.py:122-131: column sums of the OTHER factor
    kl = ctx->colsum + (which == 0 ? d.R : 0);
    rc = which == 0 ? factor_colsum(H, d.B, d.R, d.h_inner(), ctx->cs_scratch, ctx->cs_scratch_floats, kl, st)
                    : factor_colsum(W, d.C, d.R, d.w_inner(), ctx->cs_scratch, ctx->cs_scratch_floats, kl, st);
  } else {
    rc = which == 0 ? nmfd_wgrad(d, ctx->Pp, H, ctx->den, nsplit, st) : nmfd_dgrad(d, ctx->Pp, W, ctx->den, nsplit, st);
  }
  if (rc) return rc;
  a.num = ctx->num; a.den = beta == 1.0 ? nullptr : ctx->den; a.nchunks = nsplit; a.kl_den = kl;
  return 0;
}

static int nmfd_update(nmfb200_ctx* ctx, const float* W, const float* H, int which, float* param, double beta, double gamma,
                       double l1_reg, double l2_reg, cudaStream_t st) {
  ApplyArgs a; bool tc;
  int rc = nmfd_terms(ctx, W, H, which, beta, a, &tc, st);
  if (rc) return rc;
  a.param = param; a.gamma = (float)gamma; a.l1 = (float)l1_reg; a.l2 = (float)l2_reg;
  if (tc) a.absmax_bits = tc_nmfd_begin_update(ctx->tcd, which, st);
  return apply_update(a, st);
}

int nmfb200_nmfd_update_w(nmfb200_ctx* ctx, float* W, const float* H, double beta, double gamma, double l1_reg,
                          double l2_reg, void* stream) {
  CTX_GUARD(ctx, 1);
  if (!ctx->has_target) return fail(NMFB200_ERR_STATE, "set_target has not been called");
  if (!W || !H) return fail(NMFB200_ERR_INVALID, "null factor pointer");
  return nmfd_update(ctx, W, H, 0, W, beta, gamma, l1_reg, l2_reg, (cudaStream_t)stream);
}

int nmfb200_nmfd_update_h(nmfb200_ctx* ctx, const float* W, float* H, double beta, double gamma, double l1_reg,
                          double l2_reg, void* stream) {
  CTX_GUARD(ctx, 1);
  if (!ctx->has_target) return fail(NMFB200_ERR_STATE, "set_target has not been called");
  if (!W || !H) return fail(NMFB200_ERR_INVALID, "null factor pointer");
  return nmfd_update(ctx, W, H, 1, H, beta, gamma, l1_reg, l2_reg, (cudaStream_t)stream);
}

int nmfb200_nmfd_sync_factors(nmfb200_ctx* ctx) {
  CTX_GUARD(ctx, 1);
  if (ctx->tcd) tc_nmfd_mark_dirty(ctx->tcd);
  return 0;
}

int64_t nmfb200_nmfd_raw_terms_numel(const nmfb200_ctx* ctx, int which, double beta) {
  if (!ctx || ctx->kind != 1 || (which != 0 && which != 1)) return -1;
  const NmfdShape& d = ctx->d;
  const int64_t n = (int64_t)(which == 0 ? d.C : d.B) * d.R * (which == 0 ? d.w_inner() : d.h_inner());
  return beta == 1.0 ? n + d.R : 2 * n;
}

int nmfb200_nmfd_raw_terms(nmfb200_ctx* ctx, const float* W, const float* H, int which, double beta, float* out,
                           void* stream) {
  CTX_GUARD(ctx, 1);
  if (!ctx->has_target) return fail(NMFB200_ERR_STATE, "set_target has not been called");
  if (!W || !H || !out || (which != 0 && which != 1)) return fail(NMFB200_ERR_INVALID, "bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  ApplyArgs a; bool tc;
  int rc = nmfd_terms(ctx, W, H, which, beta, a, &tc, st);
  if (rc) return rc;
  rc = raw_sum(a, out, a.den ? out + a.numel : nullptr, st);
  if (rc) return rc;
  if (beta == 1.0)
    NMF_CUDA_CHECK(cudaMemcpyAsync(out + a.numel, a.kl_den, (size_t)ctx->d.R * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return 0;
}

int nmfb200_nmfd_loss(nmfb200_ctx* ctx, const float* W, const float* H, double beta, double* loss_dev,
                      void* stream) {
  CTX_GUARD(ctx, 1);
  if (!ctx->has_target) return fail(NMFB200_ERR_STATE, "set_target has not been called");
  if (!W || !H || !loss_dev) return fail(NMFB200_ERR_INVALID, "null pointer");
  if (nmfd_use_tc(ctx, beta)) return tc_nmfd_recon(ctx->tcd, ctx->V, W, H, true, loss_dev, (cudaStream_t)stream);
  return nmfd_recon_phi(ctx->d, ctx->V, W, H, beta, nullptr, nullptr, ctx->loss_blocks, ctx->loss_max_blocks,
                        loss_dev, (cudaStream_t)stream);
}

int nmfb200_hoyer_project(int device, float* x, int64_t outer, int64_t D, int64_t inner, const float* k1, const float* k2,
                          void* zeroed_ws, void* stream) {
  if (!x || !k1 || !k2 || !zeroed_ws) return fail(NMFB200_ERR_INVALID, "null pointer");
  if (outer < 1 || inner < 1 || D < 1 || D > 0x7fffffff) return fail(NMFB200_ERR_INVALID, "bad shape");
  DeviceGuard guard(device);
  if (!guard.ok) return fail(NMFB200_ERR_CUDA, "cannot select the device");
  return hoyer_project(x, outer, (int)D, inner, k1, k2, (unsigned char*)zeroed_ws, (cudaStream_t)stream);
}

}  // extern "C"
