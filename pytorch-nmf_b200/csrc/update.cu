// Ratio stage of the multiplicative update (nmf.py:78-92) and the small reductions around it.
#include "common.cuh"

namespace nmfb200 {

namespace {

__global__ void __launch_bounds__(256)
apply_update_kernel(ApplyArgs a) {
  const int64_t idx = (int64_t)blockIdx.x * 256 + threadIdx.x;
  float newv = 0.f;
  if (idx < a.numel) {
    const int64_t row = idx / a.rowlen;
    const int64_t col = idx - row * a.rowlen;
    const int64_t off = row * a.ldp + col;
    const int r = (int)((idx / a.inner) % a.R);
    float num = 0.f;
    for (int ch = 0; ch < a.nchunks; ++ch) num += a.num[ch * a.chunk_stride + off];
    if (a.kappa) num = fmaf(*a.kappa, a.kappa_vec[r], num);
    const float p = a.param[idx];
    float pos;
    if (a.den) {
      float den = 0.f;
      for (int ch = 0; ch < a.nchunks; ++ch) den += a.den[ch * a.chunk_stride + off];
      pos = fmaxf(den, 0.f) + kEps;                          // nmf.py:83
    } else {
      pos = a.kl_den[r];                                     // nmf.py:368-369 / :381-382 (no relu, no eps)
    }
    newv = mu_step(p, num, pos, a.l1, a.l2, a.gamma);
    a.param[idx] = newv;
  }
  if (a.absmax_bits) {          // one atomic per block: tens of thousands of same-address atomics serialise in L2
    __shared__ float wmax[8];
    float m = newv;
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int i = 1; i < 8; ++i) m = fmaxf(m, wmax[i]);
      if (m > 0.f) atomicMax(a.absmax_bits, __float_as_uint(m));
    }
  }
}

// The ratio stage's inputs without the ratio stage: the summed partials (+ the centring term), nothing clamped.
__global__ void __launch_bounds__(256)
raw_sum_kernel(ApplyArgs a, float* __restrict__ num_out, float* __restrict__ den_out) {
  const int64_t idx = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (idx >= a.numel) return;
  const int64_t row = idx / a.rowlen;
  const int64_t off = row * a.ldp + (idx - row * a.rowlen);
  float num = 0.f;
  for (int ch = 0; ch < a.nchunks; ++ch) num += a.num[ch * a.chunk_stride + off];
  if (a.kappa) num = fmaf(*a.kappa, a.kappa_vec[(int)((idx / a.inner) % a.R)], num);
  num_out[idx] = num;
  if (den_out) {
    float den = 0.f;
    for (int ch = 0; ch < a.nchunks; ++ch) den += a.den[ch * a.chunk_stride + off];
    den_out[idx] = den;
  }
}

// stage 1 for inner == 1: x is (outer, R) row-major; block b sums a row slab.
__global__ void __launch_bounds__(256)
colsum_rows_kernel(const float* __restrict__ x, int64_t outer, int R, int64_t rows_per_block,
                   float* __restrict__ partial) {
  __shared__ float sh[256];
  const int tid = threadIdx.x;
  const int ng = 256 / R > 0 ? 256 / R : 1;      // row groups (R <= 256)
  const int g = tid / R, r = tid - g * R;
  const int64_t row0 = (int64_t)blockIdx.x * rows_per_block;
  const int64_t row1 = min(outer, row0 + rows_per_block);
  float acc = 0.f;
  if (g < ng)
    for (int64_t row = row0 + g; row < row1; row += ng) acc += x[row * R + r];
  sh[tid] = acc;
  __syncthreads();
  if (tid < R) {
    float t = 0.f;
    for (int k = 0; k < ng; ++k) t += sh[k * R + tid];
    partial[(int64_t)blockIdx.x * R + tid] = t;
  }
}

// stage 1 for inner > 1: one block per (o, r) run of `inner` contiguous elements.
__global__ void __launch_bounds__(256)
colsum_runs_kernel(const float* __restrict__ x, int64_t inner, float* __restrict__ partial) {
  __shared__ float sh[8];
  const float* run = x + (int64_t)blockIdx.x * inner;
  float acc = 0.f;
  for (int64_t i = threadIdx.x; i < inner; i += 256) acc += run[i];
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int k = 0; k < 8; ++k) t += sh[k];
    partial[blockIdx.x] = t;      // index o*R + r
  }
}

__global__ void colsum_final_kernel(const float* __restrict__ partial, int64_t nb, int R, float* __restrict__ sums) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  float t = 0.f;
  for (int64_t b = 0; b < nb; ++b) t += partial[b * R + r];
  sums[r] = t;
}

__device__ __forceinline__ float nan_min(float a, float b) { return (a != a || b != b) ? NAN : fminf(a, b); }
__device__ __forceinline__ float nan_max(float a, float b) { return (a != a || b != b) ? NAN : fmaxf(a, b); }

// NaN-sticky min / max so that a NaN in V fails fit()'s non-negativity assertion like torch.all(V >= 0) does
__global__ void __launch_bounds__(256)
minmax_stage1(const float* __restrict__ V, int64_t rows, int64_t cols, int64_t ld, float* __restrict__ scratch) {
  __shared__ float smin[8], smax[8];
  float mn = INFINITY, mx = -INFINITY;
  const int64_t total = rows * cols;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < total; i += (int64_t)gridDim.x * 256) {
    int64_t r = i / cols, c = i - r * cols;
    float v = V[r * ld + c];
    mn = nan_min(mn, v);
    mx = nan_max(mx, v);
  }
  for (int o = 16; o > 0; o >>= 1) {
    mn = nan_min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = nan_max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) { smin[threadIdx.x >> 5] = mn; smax[threadIdx.x >> 5] = mx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 1; k < 8; ++k) { mn = nan_min(mn, smin[k]); mx = nan_max(mx, smax[k]); }
    scratch[blockIdx.x] = mn;
    scratch[1024 + blockIdx.x] = mx;
  }
}

__global__ void minmax_stage2(const float* __restrict__ scratch, int nb, float* __restrict__ mm) {
  if (threadIdx.x != 0) return;
  float mn = INFINITY, mx = -INFINITY;
  for (int k = 0; k < nb; ++k) { mn = nan_min(mn, scratch[k]); mx = nan_max(mx, scratch[1024 + k]); }
  mm[0] = mn;
  mm[1] = mx;
}

}  // namespace

// Four consecutive elements per thread (same row, same component: inner % 4 == 0), 16-byte loads of the parameter and of every
// partial slab.  Same arithmetic per element as apply_update_kernel.
__global__ void __launch_bounds__(256)
apply_update_vec4_kernel(ApplyArgs a) {
  const int64_t idx = ((int64_t)blockIdx.x * 256 + threadIdx.x) * 4;
  float m = 0.f;
  if (idx < a.numel) {
    const int64_t row = idx / a.rowlen;
    const int64_t off = row * a.ldp + (idx - row * a.rowlen);
    const int r = (int)((idx / a.inner) % a.R);
    float4 num = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int ch = 0; ch < a.nchunks; ++ch) {
      const float4 t = *reinterpret_cast<const float4*>(a.num + ch * a.chunk_stride + off);
      num.x += t.x; num.y += t.y; num.z += t.z; num.w += t.w;
    }
    float4 den = make_float4(0.f, 0.f, 0.f, 0.f);
    if (a.den) {
      for (int ch = 0; ch < a.nchunks; ++ch) {
        const float4 t = *reinterpret_cast<const float4*>(a.den + ch * a.chunk_stride + off);
        den.x += t.x; den.y += t.y; den.z += t.z; den.w += t.w;
      }
    }
    const float klden = a.den ? 0.f : a.kl_den[r];
    float4 p = *reinterpret_cast<const float4*>(a.param + idx);
    auto one = [&](float pv, float n, float d) {
      if (a.kappa) n = fmaf(*a.kappa, a.kappa_vec[r], n);
      const float pos = a.den ? fmaxf(d, 0.f) + kEps : klden;   // nmf.py:83 / :368-369
      return mu_step(pv, n, pos, a.l1, a.l2, a.gamma);
    };
    p.x = one(p.x, num.x, den.x); p.y = one(p.y, num.y, den.y); p.z = one(p.z, num.z, den.z); p.w = one(p.w, num.w, den.w);
    *reinterpret_cast<float4*>(a.param + idx) = p;
    m = fmaxf(fmaxf(p.x, p.y), fmaxf(p.z, p.w));
  }
  if (a.absmax_bits) {
    __shared__ float wmax[8];
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int i = 1; i < 8; ++i) m = fmaxf(m, wmax[i]);
      if (m > 0.f) atomicMax(a.absmax_bits, __float_as_uint(m));
    }
  }
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int apply_update(const ApplyArgs& a, cudaStream_t st) {
  if (a.numel <= 0) return 0;
  const bool vec4 = a.inner % 4 == 0 && a.rowlen % 4 == 0 && a.ldp % 4 == 0 && a.numel % 4 == 0 &&
                    (a.nchunks == 1 || a.chunk_stride % 4 == 0) && aligned16(a.param) && aligned16(a.num) &&
                    (!a.den || aligned16(a.den));
  if (vec4)
    apply_update_vec4_kernel<<<(unsigned)ceil_div(a.numel / 4, 256), 256, 0, st>>>(a);
  else
    apply_update_kernel<<<(unsigned)ceil_div(a.numel, 256), 256, 0, st>>>(a);
  NMF_LAUNCH_CHECK();
  return 0;
}

int raw_sum(const ApplyArgs& a, float* num_out, float* den_out, cudaStream_t st) {
  if (a.numel <= 0) return 0;
  raw_sum_kernel<<<(unsigned)ceil_div(a.numel, 256), 256, 0, st>>>(a, num_out, a.den ? den_out : nullptr);
  NMF_LAUNCH_CHECK();
  return 0;
}

static int64_t colsum_blocks(int64_t outer, int64_t inner) {
  if (inner > 1) return outer;   // one per (o, r) run, x R below
  int64_t nb = ceil_div(outer, 64);
  return nb > 1024 ? 1024 : (nb < 1 ? 1 : nb);
}

int64_t colsum_scratch_floats(int64_t outer, int R, int64_t inner) { return colsum_blocks(outer, inner) * R; }

int factor_colsum(const float* x, int64_t outer, int R, int64_t inner, float* scratch, int64_t scratch_floats,
                  float* sums, cudaStream_t st) {
  if (R > 256) { set_error("factor_colsum: rank must be <= 256"); return 1; }
  const int64_t nb = colsum_blocks(outer, inner);
  if (nb * R > scratch_floats) { set_error("factor_colsum: scratch too small"); return 1; }
  if (inner > 1) {
    colsum_runs_kernel<<<(unsigned)(outer * R), 256, 0, st>>>(x, inner, scratch);
  } else {
    const int64_t rpb = ceil_div(outer, nb);
    colsum_rows_kernel<<<(unsigned)nb, 256, 0, st>>>(x, outer, R, rpb, scratch);
  }
  NMF_LAUNCH_CHECK();
  colsum_final_kernel<<<(unsigned)ceil_div(R, 64), 64, 0, st>>>(scratch, nb, R, sums);
  NMF_LAUNCH_CHECK();
  return 0;
}

int matrix_minmax(const float* V, int64_t rows, int64_t cols, int64_t ld, float* scratch2048, float* mm,
                  cudaStream_t st) {
  int64_t nb = ceil_div(rows * cols, 256 * 16);
  if (nb > 1024) nb = 1024;
  if (nb < 1) nb = 1;
  minmax_stage1<<<(unsigned)nb, 256, 0, st>>>(V, rows, cols, ld, scratch2048);
  NMF_LAUNCH_CHECK();
  minmax_stage2<<<1, 32, 0, st>>>(scratch2048, (int)nb, mm);
  NMF_LAUNCH_CHECK();
  return 0;
}

}  // namespace nmfb200
