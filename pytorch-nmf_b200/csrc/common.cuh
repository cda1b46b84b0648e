// Shared declarations for the libnmf_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

namespace nmfb200 {

// torchnmf/constants.py:3 -- float32 machine epsilon, 2^-23
constexpr float kEps = 1.1920928955078125e-07f;

// beta-divergence branch of nmf.py:61-74 / metrics.py:60-96
enum BetaMode : int { kKL = 0, kEU = 1, kIS = 2, kGeneric = 3 };
inline BetaMode beta_mode(double beta) {
  if (beta == 1.0) return kKL;
  if (beta == 2.0) return kEU;
  if (beta == 0.0) return kIS;
  return kGeneric;
}

void set_error(const std::string& msg);
void count_launch();

#define NMF_CUDA_CHECK(expr)                                                              \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      nmfb200::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));             \
      return 2;                                                                           \
    }                                                                                     \
  } while (0)

#define NMF_LAUNCH_CHECK()                                                                \
  do {                                                                                    \
    nmfb200::count_launch();                                                              \
    cudaError_t _e = cudaGetLastError();                                                  \
    if (_e != cudaSuccess) {                                                              \
      nmfb200::set_error(std::string("kernel launch: ") + cudaGetErrorString(_e));        \
      return 2;                                                                           \
    }                                                                                     \
  } while (0)

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline int64_t round_up(int64_t a, int64_t b) { return ceil_div(a, b) * b; }

// The element step of the multiplicative update (nmf.py:78-92) once the numerator `num` and the denominator `pos` of
// element `v` are formed: v ((relu(num) + eps) / (pos [+ l1] [+ l2 v]))^gamma.  Each ratio-stage kernel sums its own
// partials and forms `pos` (relu(den) + eps, or the KL column sum); the tail is this one.
__device__ __forceinline__ float mu_step(float v, float num, float pos, float l1, float l2, float gamma) {
  const float neg = fmaxf(num, 0.f) + kEps;              // nmf.py:78
  if (l1 > 0.f) pos += l1;                               // nmf.py:85-86
  if (l2 > 0.f) pos = fmaf(l2, v, pos);                  // nmf.py:87-88
  float mult = neg / pos;                                // nmf.py:89
  if (gamma != 1.0f) mult = powf(mult, gamma);           // nmf.py:90-91
  return v * mult;                                       // nmf.py:92
}

// ------------------------------------------------------------------------------------------
// Launch wrappers implemented in the .cu files (all asynchronous on `st`, return 0 / error code)
// ------------------------------------------------------------------------------------------

// simt_nmf.cu ------------------------------------------------------------------------------
// Partial contractions of one factor update on CUDA cores, fp32:
//   S = F G^T (Mr x Nc),  (Pn, Pp) = phi_beta(Vm, S)          [nmf.py:61-74]
//   num[ch][m][r] = sum_{c in chunk ch} Pn[m,c] G[c,r]          [nmf.py:77]
//   den[ch][m][r] = sum_{c in chunk ch} Pp[m,c] G[c,r]          [nmf.py:82, beta != 1 only]
// Vm[m,c] = V[m*ldv + c] (trans = 0) or V[c*ldv + m] (trans = 1).
int simt_nmf_contract(const float* V, int64_t ldv, int trans, const float* F, const float* G,
                      int64_t Mr, int64_t Nc, int R, double beta, int nchunks,
                      float* num, float* den, int64_t ldp, int64_t chunk_stride, cudaStream_t st);
// beta_div(F G^T, Vm) accumulated into block partials then *loss_dev (double).  v_const is unused here.
int simt_nmf_loss(const float* V, int64_t ldv, const float* F, const float* G, int64_t Mr, int64_t Nc,
                  int R, double beta, double* block_partials, int max_blocks, double* loss_dev,
                  cudaStream_t st);
int simt_nmf_max_blocks(int64_t Mr, int64_t Nc);

// update.cu --------------------------------------------------------------------------------
// nmf.py:78-92 on a flattened parameter of `numel` elements whose rank index is
// r = (idx / inner) % R.   num/den are sums over `nchunks` partial slabs (stride chunk_stride,
// row pitch ldp for a (rows x R*inner) view: element idx -> (idx / rowlen) * ldp + idx % rowlen).
struct ApplyArgs {
  float* param; int64_t numel; int R; int64_t inner; int64_t rowlen;
  const float* num; const float* den; int nchunks; int64_t chunk_stride; int64_t ldp;
  const float* kl_den;     // [R] when beta == 1 (den == nullptr)
  float gamma, l1, l2;
  unsigned int* absmax_bits;  // optional: atomicMax of the updated values (non-negative floats)
  const float* kappa;         // optional (with kappa_vec): the partials hold sum (P - kappa) G; num += *kappa * kappa_vec[r]
  const float* kappa_vec;     // [R]
};
int apply_update(const ApplyArgs& a, cudaStream_t st);
// num_out[i] (and den_out[i] when a.den) = what the ratio stage would read for element i: summed partials + centring term
int raw_sum(const ApplyArgs& a, float* num_out, float* den_out, cudaStream_t st);
// sums[r] = sum over all other dims of x viewed as (outer, R, inner); deterministic two-stage.
int factor_colsum(const float* x, int64_t outer, int R, int64_t inner, float* scratch, int64_t scratch_floats,
                  float* sums, cudaStream_t st);
int64_t colsum_scratch_floats(int64_t outer, int R, int64_t inner);
// min / max of a strided fp32 matrix (fit()'s validation), results in mm[0..1]
int matrix_minmax(const float* V, int64_t rows, int64_t cols, int64_t ld, float* scratch2048, float* mm,
                  cudaStream_t st);
// *out = sum of n doubles in fixed order (single block)
int sum_partials(const double* p, int n, double* out, cudaStream_t st);

// project.cu -------------------------------------------------------------------------------
// Hoyer's projection (nmf.py:21-49) of every slice x[:, j, :] of x viewed as (outer, D, inner) onto {v >= 0, |v|_1 = k1[j],
// |v|_2^2 = k2[j]}, in place; zeroed_ws: D * outer * inner bytes of scratch.
int hoyer_project(float* x, int64_t outer, int D, int64_t inner, const float* k1, const float* k2,
                  unsigned char* zeroed_ws, cudaStream_t st);

// sparse_nmf.cu ----------------------------------------------------------------------------
// Sparse-target NMF for beta 1 and 2 (nmf.py:603-638): update terms at the non-zeros of V only, one warp per compressed segment.
int sparse_numerator(const int64_t* ptr, const int64_t* idx, const float* val, const float* Fself, const float* Fother,
                     int R, int64_t nseg, double beta, float* out, cudaStream_t st);
int sparse_gram(const float* F, int64_t rows, int R, float* part, float* out, cudaStream_t st);          // out = F^T F (R x R)
int64_t sparse_gram_part_floats(int R);
int sparse_rows_times_gram(const float* F, const float* G, int64_t rows, int R, float* out, cudaStream_t st);
int sparse_loss(const int64_t* crow, const int64_t* col, const float* val, const float* H, const float* W, int R, int64_t N,
                double beta, const float* pos_a, const float* pos_b, double v_norm, double* loss_part, double* loss_dev,
                cudaStream_t st);
int sparse_loss_blocks(int64_t N);

// nmfd.cu ----------------------------------------------------------------------------------
// L, T, Lin are the sizes along the LAST (contiguous) axis; NMF2D / NMF3D (nmf.py:782-942) add up to two outer axes of the
// target (X1, X2), of the kernel (T1, T2) and of H (X - T + 1).  The outer axes are loops around the same sliding GEMMs.
struct NmfdShape {
  int B, C, L, R, T, Lin;
  int X1 = 1, X2 = 1, T1 = 1, T2 = 1;
  __host__ __device__ int J1() const { return X1 - T1 + 1; }
  __host__ __device__ int J2() const { return X2 - T2 + 1; }
  __host__ __device__ int64_t v_inner() const { return (int64_t)X1 * X2 * L; }        // target elements per (b, c)
  __host__ __device__ int64_t w_inner() const { return (int64_t)T1 * T2 * T; }        // kernel elements per (c, r)
  __host__ __device__ int64_t h_inner() const { return (int64_t)J1() * J2() * Lin; }  // activation elements per (b, r)
  __host__ __device__ bool one_d() const { return X1 == 1 && X2 == 1 && T1 == 1 && T2 == 1; }
};
// WH = conv(H, W); writes Pn (and Pp when beta != 1) (B,C,L) or, when loss_blocks != nullptr,
// reduces beta_div(WH, V) instead.
int nmfd_recon_phi(const NmfdShape& s, const float* V, const float* W, const float* H, double beta,
                   float* Pn, float* Pp, double* loss_blocks, int max_blocks, double* loss_dev,
                   cudaStream_t st);
int nmfd_max_blocks(const NmfdShape& s);
// out[c,r,t] = sum_{b,x} G[b,c,x] H[b,r,x-t]   (x, t multi-indices over up to three axes)
int nmfd_wgrad(const NmfdShape& s, const float* G, const float* H, float* out, int nsplit, cudaStream_t st);   // out[split][C,R,T]
int nmfd_wgrad_nsplit(const NmfdShape& s);
// out[split][b,r,j] = sum_{c in split, t} W[c,r,t] G[b,c,j+t]   (j, t multi-indices)
int nmfd_dgrad(const NmfdShape& s, const float* G, const float* W, float* out, int nsplit, cudaStream_t st);
int nmfd_dgrad_nsplit(const NmfdShape& s);

}  // namespace nmfb200
