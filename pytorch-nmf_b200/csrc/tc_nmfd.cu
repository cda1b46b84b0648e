// NMFD (1-D convolutive NMF, nmf.py:776-779) on tcgen05 tensor cores for beta = 1: the three contractions of an update as
// im2col-free SLIDING GEMMs.
//
//   recon : S[c, l]     = sum_{r,t} W[c,r,t] H[r, l-t]           then the ratio epilogue  P~ = (V / (S + eps) - kappa) 2^p  (fp16)
//   wgrad : gW[c, r, t] = sum_l  P~[c, l] H[r, l-t]              (W update: numerator = gW / 2^.. + kappa colsum(H))
//   dgrad : gH[r, j]    = sum_{c,t} W[c,r,t] P~[c, j+t]          (H update: numerator = gH / 2^.. + kappa colsum(W))
//
// recon and dgrad use the eight-phase formulation (tcnmfd_recon2_kernel, tcnmfd_dgrad2_kernel): the big operand is the raw
// fp16 row in shared memory under an overlapping descriptor, the small one eight shifted copies of W.  wgrad
// (tcnmfd_wgrad_kernel) is a GEMM whose A operand is a plain matrix (P~, TMA, SWIZZLE_128B) and whose B operand is a
// Toeplitz matrix: row t of a 128 x 64 tile is the 64-element window of a padded row of H that starts one element earlier
// than row t - 1.  Nothing of that matrix ever exists in global memory: per k-block the TMA warp bulk-copies the
// ~200-element source window into shared memory and the eight producer warps write the 128 x 64 tile from it in the UMMA
// SWIZZLE_128B K-major layout (4-byte shared loads, one byte-permute per word for odd shifts, 16-byte stores), 2 threads
// per row.  The MMA warp issues tcgen05.mma SS on it exactly as on a TMA-written tile; the accumulator lives in TMEM; the
// epilogue warps read it back with tcgen05.ld.
//
// Scope: T <= 128 (tc_nmfd_shape_supported).  wgrad holds every shift of a (128-row c tile, component) in ONE 128 x 128
// accumulator whose columns are the shifts, and at T = 128 the eight-phase stages take about 110 KB of shared memory.
// Longer kernels run on the fp32 sliding GEMMs of nmfd.cu.
//
// Precision design = the NMF kernel's (DESIGN.md 4.2): fp16 operands with power-of-two scales, fp32 accumulation, the
// ratio tile centred on kappa = sum(V) / sum(WH) so that the K = 8192 ... 131200-term numerator sums are signed and small
// (tensor-core accumulation truncates), kappa * colsum added back in fp32 by the ratio stage (apply_update).
#include "tc_nmfd.cuh"

#include <cuda.h>

#include <algorithm>
#include <string>

#include "sm100_ptx.cuh"

namespace nmfb200 {

namespace {

constexpr int kM = 128;            // tile rows (TMEM lanes)
constexpr int kKB = 64;            // k-block: 64 fp16 = one 128-byte swizzle row
constexpr int kStages = 3;
constexpr int kWinHalfs = 256;     // source window per k-block: 128 rows + 64 columns + alignment slack (512 bytes)
constexpr int kThreads = 384;      // warp 0 TMA | warp 1 MMA | warps 2-3 idle | warps 4-11 producers (8-11 also epilogue)

struct WgradParams {
  int B, C, L, R, T;
  int Lp;                         // padded row length of Hp16 (halfs); H[b,r,j] sits at column padl + j
  int padl;
  const __half* Hp16;             // [B*R][Lp]
  const int* exps;                // {eW, eH, eP}: power-of-two exponents of W16, Hp16, P16
  float* out;                     // [nsplit][C][R][T]
  int kb_per_split;
};

struct Smem {
  static constexpr int kTile = kM * kKB * 2;                 // 16 KB
  static constexpr int kPlain = 0;
  static constexpr int kToep = kStages * kTile;
  static constexpr int kWin = 2 * kStages * kTile;
  static constexpr int kBar = kWin + kStages * kWinHalfs * 2;
  static constexpr int kNumBars = 4 * kStages + 1;           // win_full, tile_full, empty, win_read per stage + acc_full
  static constexpr int kTmemPtr = kBar + 8 * kNumBars;
  static constexpr int kTotal = kTmemPtr + 16;
};

__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(bar)
               : "memory");
}

// grid (C tiles, R, nsplit): A = P16 tile (rows c, by TMA), B = Toeplitz tile of the H row of component blockIdx.y (rows t,
// built by the producers), N = 128 shifts; split z walks k-blocks [kb_per_split z, kb_per_split (z + 1)) of (b, l)
__global__ void __launch_bounds__(kThreads, 2)
tcnmfd_wgrad_kernel(const __grid_constant__ CUtensorMap tmP, const WgradParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t raw32 = ptx::smem_u32(smem_raw);
  const uint32_t sbase = (raw32 + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (sbase - raw32);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  auto BAR = [&](int i) { return sbase + Smem::kBar + 8u * i; };
  constexpr int B_WIN = 0, B_TILE = kStages, B_EMPTY = 2 * kStages, B_WREAD = 3 * kStages, B_ACC = 4 * kStages;
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem_al + Smem::kTmemPtr);

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmP);
    for (int i = 0; i < kStages; ++i) {
      ptx::mbar_init(BAR(B_WIN + i), 1);
      ptx::mbar_init(BAR(B_TILE + i), 8);        // one arrival per producer warp
      ptx::mbar_init(BAR(B_EMPTY + i), 1);
      ptx::mbar_init(BAR(B_WREAD + i), 8);       // the 8 producer warps have read the source window of this stage
    }
    ptx::mbar_init(BAR(B_ACC), 1);
    ptx::fence_barrier_init();
    ptx::fence_proxy_async();
  }
  if (warp == 1) {
    ptx::tmem_alloc(sbase + Smem::kTmemPtr, 128);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = *tmem_ptr_smem;

  // ---- what this CTA computes, as a list of k-blocks: (P16 tile coordinates, H row, window start) ------------------------
  const int kb0 = blockIdx.z * p.kb_per_split;
  const int lkb = (p.L + kKB - 1) / kKB;                    // k-blocks per batch element
  const int nkb = max(0, min(p.kb_per_split, p.B * lkb - kb0));
  // per k-block: returns the P16 tile's TMA coordinates (x = column, y = row), the H row pointer and the index of the H
  // element that row 0 / column 0 of the Toeplitz tile reads; row t reads one element earlier than row t - 1
  auto kblock = [&](int kb, int& px, int& py, const __half*& src, int& e0) {
    const int g = kb0 + kb, b = g / lkb, lk = g - b * lkb;
    px = lk * kKB; py = b * p.C + blockIdx.x * kM;
    src = p.Hp16 + ((int64_t)b * p.R + blockIdx.y) * p.Lp;
    e0 = p.padl + lk * kKB;                                 // row t reads H[l - t]: e0 - t
  };
  // window = source elements [wbeg, wbeg + kWinHalfs), wbeg 8-aligned and <= the smallest index any row reads
  auto win_begin = [&](int e0) { return (e0 - (kM - 1)) & ~7; };

  if (warp == 0) {
    // =========================== TMA: P16 tile + source window per k-block ===========================================
    if (lane == 0) {
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % kStages, ph = (kb / kStages) & 1;
        ptx::mbar_wait(BAR(B_EMPTY + s), ph ^ 1);      // the MMAs that read this stage's tiles have completed ...
        ptx::mbar_wait(BAR(B_WREAD + s), ph ^ 1);      // ... and every producer warp has read its source window
        int px, py, e0; const __half* src;
        kblock(kb, px, py, src, e0);
        ptx::mbar_expect_tx(BAR(B_WIN + s), (uint32_t)Smem::kTile + kWinHalfs * 2);
        ptx::tma_load_2d(&tmP, BAR(B_WIN + s), sbase + Smem::kPlain + s * Smem::kTile, px, py);
        bulk_copy_g2s(sbase + Smem::kWin + s * kWinHalfs * 2, src + win_begin(e0), kWinHalfs * 2, BAR(B_WIN + s));
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer ==========================================================================
    const uint32_t idesc = ptx::idesc_f16(kM, 128, 0, 0);
    constexpr uint32_t descHi = ptx::smem_desc_hi_sw128(1024);
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % kStages, ph = (kb / kStages) & 1;
      if (lane == 0) {
        ptx::mbar_wait(BAR(B_WIN + s), ph);       // P16 tile landed (TMA -> this thread)
        ptx::mbar_wait(BAR(B_TILE + s), ph);      // Toeplitz tile written by the 8 producer warps
      }
      __syncwarp();
      ptx::tc_fence_after();
      const uint32_t plain = sbase + Smem::kPlain + s * Smem::kTile, toep = sbase + Smem::kToep + s * Smem::kTile;
      if (ptx::elect_one()) {
#pragma unroll
        for (int ks = 0; ks < kKB / 16; ++ks) {
          const uint32_t alo = ptx::smem_desc_lo(plain, 16) + 2 * ks, blo = ptx::smem_desc_lo(toep, 16) + 2 * ks;
          ptx::mma_ss(tmem, ptx::make_desc(alo, descHi), ptx::make_desc(blo, descHi), idesc, (kb | ks) ? 1u : 0u);
        }
        ptx::mma_commit(BAR(B_EMPTY + s));
        if (kb == nkb - 1) ptx::mma_commit(BAR(B_ACC));
      }
      __syncwarp();
    }
  } else if (warp >= 4) {
    // =========================== Toeplitz producers: 8 warps, 2 threads per tile row ==================================
    const int pt = threadIdx.x - 128;              // 0..255
    const int row = pt >> 1, half = pt & 1;        // this thread writes columns [32 half, 32 half + 32) of its row
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % kStages, ph = (kb / kStages) & 1;
      int px, py, e0; const __half* src;
      kblock(kb, px, py, src, e0);
      const int off = e0 - row - win_begin(e0) + 32 * half;             // first window element this thread reads (>= 0)
      ptx::mbar_wait(BAR(B_WIN + s), ph);                               // window (and P16 tile) landed
      const uint32_t win = sbase + Smem::kWin + s * kWinHalfs * 2 + (uint32_t)(off >> 1) * 4;
      uint32_t w[17];
#pragma unroll
      for (int i = 0; i < 17; ++i) asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w[i]) : "r"(win + 4 * i));
      const uint32_t sel = (off & 1) ? 0x5432u : 0x3210u;                // odd start: take the upper half of w[i] and the lower of w[i+1]
      uint32_t o[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) o[i] = __byte_perm(w[i], w[i + 1], sel);
      const uint32_t dst = sbase + Smem::kToep + s * Smem::kTile + row * 128;
#pragma unroll
      for (int c16 = 0; c16 < 4; ++c16) {
        const uint32_t chunk = (uint32_t)(4 * half + c16) ^ (uint32_t)(row & 7);      // SWIZZLE_128B
        asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};"
                     ::"r"(dst + (chunk << 4)), "r"(o[4 * c16]), "r"(o[4 * c16 + 1]), "r"(o[4 * c16 + 2]), "r"(o[4 * c16 + 3])
                     : "memory");
      }
      ptx::fence_proxy_async();                    // generic-proxy stores -> visible to the tensor core (async proxy)
      __syncwarp();
      if (lane == 0) { ptx::mbar_arrive(BAR(B_TILE + s)); ptx::mbar_arrive(BAR(B_WREAD + s)); }
    }
    if (warp >= 8) {
      // =========================== epilogue (warps 8-11 = TMEM lane quarters 0-3): row c, columns t ==================
      const int q = warp & 3, r128 = q * 32 + lane;
      const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
      ptx::mbar_wait(BAR(B_ACC), 0);
      ptx::tc_fence_after();
      const float sc = exp2f(-(float)(p.exps[2] + p.exps[1]));
      const int c = blockIdx.x * kM + r128, r = blockIdx.y;
      float* dst = p.out + (((int64_t)blockIdx.z * p.C + (c < p.C ? c : 0)) * p.R + r) * p.T;    // [split][C][R][T]
      const bool vec = (p.T & 3) == 0;
#pragma unroll 1
      for (int j = 0; j < kM / 16; ++j) {
        uint32_t sr[16];
        ptx::tmem_ld16(tmem + lane_addr + j * 16, sr);
        ptx::tc_wait_ld();
        if (c < p.C && j * 16 < p.T) {
          if (vec && j * 16 + 16 <= p.T) {
#pragma unroll
            for (int i = 0; i < 16; i += 4)
              *reinterpret_cast<float4*>(dst + j * 16 + i) = make_float4(__uint_as_float(sr[i]) * sc, __uint_as_float(sr[i + 1]) * sc,
                                                                         __uint_as_float(sr[i + 2]) * sc, __uint_as_float(sr[i + 3]) * sc);
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i)
              if (j * 16 + i < p.T) dst[j * 16 + i] = __uint_as_float(sr[i]) * sc;
          }
        }
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem, 128);
}

// ---- dgrad, second formulation: no Toeplitz tile is built at all ---------------------------------------------------------
//   gH[r, 8q + s] = sum_c sum_u  P[c, 8q + u] * Ws[c, (r, s), u],      Ws[c, (r, s), u] = W[c, r, u - s]  (0 <= u - s < T)
// With the output position split as j = 8q + s, the eight phases s move into the SMALL operand (eight shifted copies of W,
// prepared once per update: N = (r, s) = 128 columns for 16 components), and the rows q of the big operand become windows
// of P that start 8 elements = 16 BYTES apart: exactly the row pitch of a SWIZZLE_NONE K-major core matrix.  The A operand
// of tcgen05.mma is therefore the raw fp16 row of P in shared memory, addressed by a descriptor whose core matrices overlap
// (leading byte offset 16, stride byte offset 128): one 2.4 KB bulk copy per (c, 1024 output positions) instead of a
// 128 x 64 tile per 64 shifts, and every MMA is a full-rate 128 x 128 x 16.  B = Ws tiles by TMA (SWIZZLE_128B).
// grid (ceil(Lin / 2048), nsplit over c, B * ngroups);  2 accumulators (2 x 1024 output positions) share every B tile.
constexpr int kD2Threads = 256;     // warp 0 TMA | warp 1 MMA | warps 4-7 epilogue
constexpr int kD2Stages = 2;     // per CTA; two CTAs per SM (one in its epilogue while the other runs its main loop)
constexpr int kD2Q = 2;             // q tiles (accumulators) per CTA

struct Dgrad2Params {
  int B, C, R, Lin, Lq, Tq, ngroups, nks;      // nks: 16-wide k-steps that carry shifts u <= T + 6
  const __half* P16;
  const int* exps;
  float* out;                       // [nsplit][B][R][Lin]
  int c_per_split;
};

__global__ void __launch_bounds__(kD2Threads, 2)
tcnmfd_dgrad2_kernel(const __grid_constant__ CUtensorMap tmWs, const Dgrad2Params p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t raw32 = ptx::smem_u32(smem_raw);
  const uint32_t sbase = (raw32 + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (sbase - raw32);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkk = p.Tq / kKB;                                   // B tiles (64 columns of u each) per c
  const uint32_t seg_bytes = (uint32_t)(1024 + p.Tq) * 2;       // P[c][8 q0 .. 8 q0 + 1024 + Tq)
  const uint32_t seg_pitch = (seg_bytes + 127u) & ~127u;
  const uint32_t stage_bytes = (uint32_t)nkk * Smem::kTile + kD2Q * seg_pitch;
  const uint32_t bar0 = sbase + kD2Stages * ((stage_bytes + 1023u) & ~1023u);
  auto STAGE = [&](int s) { return sbase + (uint32_t)s * ((stage_bytes + 1023u) & ~1023u); };
  auto BAR = [&](int i) { return bar0 + 8u * i; };
  constexpr int B_FULL = 0, B_EMPTY = kD2Stages, B_ACC = 2 * kD2Stages;
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem_al + (bar0 - sbase) + 8 * (2 * kD2Stages + 1));
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmWs);
    for (int i = 0; i < kD2Stages; ++i) { ptx::mbar_init(BAR(B_FULL + i), 1); ptx::mbar_init(BAR(B_EMPTY + i), 1); }
    ptx::mbar_init(BAR(B_ACC), 1);
    ptx::fence_barrier_init();
    ptx::fence_proxy_async();
  }
  if (warp == 1) {
    ptx::tmem_alloc(bar0 + 8 * (2 * kD2Stages + 1), 256);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = *tmem_ptr_smem;
  const int b = blockIdx.z / p.ngroups, grp = blockIdx.z - b * p.ngroups;
  const int c0 = blockIdx.y * p.c_per_split, c1 = min(p.C, c0 + p.c_per_split);
  const int nc = max(0, c1 - c0);
  const int j0 = blockIdx.x * (kD2Q * 1024);                    // first output position of this CTA

  if (warp == 0) {
    if (lane == 0) {
      for (int i = 0; i < nc; ++i) {
        const int s = i % kD2Stages, ph = (i / kD2Stages) & 1, c = c0 + i;
        ptx::mbar_wait(BAR(B_EMPTY + s), ph ^ 1);
        ptx::mbar_expect_tx(BAR(B_FULL + s), (uint32_t)nkk * Smem::kTile + kD2Q * seg_bytes);
        for (int kk = 0; kk < nkk; ++kk)
          ptx::tma_load_2d(&tmWs, BAR(B_FULL + s), STAGE(s) + kk * Smem::kTile, kk * kKB, (c * p.ngroups + grp) * 128);
        for (int qt = 0; qt < kD2Q; ++qt)
          bulk_copy_g2s(STAGE(s) + nkk * Smem::kTile + qt * seg_pitch,
                        p.P16 + ((int64_t)b * p.C + c) * p.Lq + j0 + qt * 1024, seg_bytes, BAR(B_FULL + s));
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = ptx::idesc_f16(kM, 128, 0, 0);
    constexpr uint32_t descHiB = ptx::smem_desc_hi_sw128(1024);
    constexpr uint32_t descHiA = ((128u >> 4) & 0x3FFFu) | (1u << 14);      // SWIZZLE_NONE, stride byte offset 128 (8 rows x 16 B)
    for (int i = 0; i < nc; ++i) {
      const int s = i % kD2Stages, ph = (i / kD2Stages) & 1;
      if (lane == 0) ptx::mbar_wait(BAR(B_FULL + s), ph);
      __syncwarp();
      ptx::tc_fence_after();
      if (ptx::elect_one()) {
        for (int qt = 0; qt < kD2Q; ++qt) {
          const uint32_t seg = STAGE(s) + nkk * Smem::kTile + qt * seg_pitch;
          for (int kst = 0; kst < p.nks; ++kst) {
            const int kk = kst >> 2, ks = kst & 3;
            // A: rows q = windows of the raw P row, 16 bytes apart; k-step = 16 elements = two core matrices 16 bytes apart
            const uint32_t alo = ptx::smem_desc_lo(seg + (uint32_t)(kst * 16) * 2, 16);
            const uint32_t blo = ptx::smem_desc_lo(STAGE(s) + kk * Smem::kTile, 16) + 2 * ks;
            ptx::mma_ss(tmem + qt * 128, ptx::make_desc(alo, descHiA), ptx::make_desc(blo, descHiB), idesc, (i | kst) ? 1u : 0u);
          }
        }
        ptx::mma_commit(BAR(B_EMPTY + s));
        if (i == nc - 1) ptx::mma_commit(BAR(B_ACC));
      }
      __syncwarp();
    }
  } else if (warp >= 4) {
    const int q = warp & 3, r128 = q * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    if (nc > 0) {
      ptx::mbar_wait(BAR(B_ACC), 0);
      ptx::tc_fence_after();
    }
    const float sc = exp2f(-(float)(p.exps[0] + p.exps[2]));
    for (int qt = 0; qt < kD2Q; ++qt) {
      const int j = j0 + qt * 1024 + 8 * r128;                   // this lane's 8 output positions
#pragma unroll 1
      for (int jj = 0; jj < 8; ++jj) {                            // 16 columns = 2 components x 8 phases
        uint32_t sr[16];
        if (nc > 0) { ptx::tmem_ld16(tmem + lane_addr + qt * 128 + jj * 16, sr); ptx::tc_wait_ld(); }
        else {
#pragma unroll
          for (int i = 0; i < 16; ++i) sr[i] = 0u;
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int r = grp * 16 + jj * 2 + h;
          if (r < p.R) {
            float* dst = p.out + (((int64_t)blockIdx.y * p.B + b) * p.R + r) * p.Lin + j;
#pragma unroll
            for (int i = 0; i < 8; ++i)
              if (j + i < p.Lin) dst[i] = __uint_as_float(sr[8 * h + i]) * sc;
          }
        }
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem, 256);
}

// ---- recon, second formulation: the same eight-phase trick on the H side ---------------------------------------------------
//   S[c, 8q + s] = sum_r sum_u  Wsh[(c, s), (r, u)] * H[r, 8q + u - A],      Wsh[(c, s), (r, u)] = W[c, r, s + A - u]
// (A = T - 1 rounded up to 8, so that the window of H that row q reads starts 16-byte aligned).  M = 16 rows c x 8 phases s
// from eight shifted copies of W (TMA, SWIZZLE_128B), N = 256 positions q = the raw padded fp16 row of H in shared memory
// through an overlapping SWIZZLE_NONE descriptor (rows 16 bytes apart): no Toeplitz tile, every MMA a 128 x 256 x 16.
// Epilogue: TMEM lane (c, s), column q  <->  S[c, 8q + s]; the eight phases of a row are neighbouring lanes, so the fp32
// reads of V and the fp16 writes of the ratio tile coalesce across lanes.
// grid (ceil(L / 2048), ceil(C / 16), B)
constexpr int kR2N = 256;

struct Recon2Params {
  int B, C, L, R, Lp, padl, Lq, Tq, A8, nks;   // nks: 16-wide k-steps that carry shifts u <= A8 + 7
  const __half* Hp16;
  __half* P16out;
  const float* V;
  const int* exps;
  const float* kappa;
  double* loss_part;
};

template <bool LOSS>
__global__ void __launch_bounds__(kD2Threads, 2)
tcnmfd_recon2_kernel(const __grid_constant__ CUtensorMap tmWsh, const Recon2Params p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t raw32 = ptx::smem_u32(smem_raw);
  const uint32_t sbase = (raw32 + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (sbase - raw32);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkk = p.Tq / kKB;
  const uint32_t seg_bytes = (uint32_t)(8 * kR2N + p.Tq) * 2;
  const uint32_t stage_pitch = ((uint32_t)nkk * Smem::kTile + seg_bytes + 1023u) & ~1023u;
  const uint32_t bar0 = sbase + kD2Stages * stage_pitch;
  auto STAGE = [&](int s) { return sbase + (uint32_t)s * stage_pitch; };
  auto BAR = [&](int i) { return bar0 + 8u * i; };
  constexpr int B_FULL = 0, B_EMPTY = kD2Stages, B_ACC = 2 * kD2Stages;
  const uint32_t tptr = bar0 + 8 * (2 * kD2Stages + 1);
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem_al + (tptr - sbase));
  double* red = reinterpret_cast<double*>(smem_al + (tptr - sbase) + 16);
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmWsh);
    for (int i = 0; i < kD2Stages; ++i) { ptx::mbar_init(BAR(B_FULL + i), 1); ptx::mbar_init(BAR(B_EMPTY + i), 1); }
    ptx::mbar_init(BAR(B_ACC), 1);
    ptx::fence_barrier_init();
    ptx::fence_proxy_async();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tptr, kR2N);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = *tmem_ptr_smem;
  const int b = blockIdx.z, cg = blockIdx.y, l0 = blockIdx.x * (8 * kR2N);

  if (warp == 0) {
    if (lane == 0) {
      for (int r = 0; r < p.R; ++r) {
        const int s = r % kD2Stages, ph = (r / kD2Stages) & 1;
        ptx::mbar_wait(BAR(B_EMPTY + s), ph ^ 1);
        ptx::mbar_expect_tx(BAR(B_FULL + s), (uint32_t)nkk * Smem::kTile + seg_bytes);
        for (int kk = 0; kk < nkk; ++kk)
          ptx::tma_load_2d(&tmWsh, BAR(B_FULL + s), STAGE(s) + kk * Smem::kTile, r * p.Tq + kk * kKB, cg * 128);
        bulk_copy_g2s(STAGE(s) + nkk * Smem::kTile, p.Hp16 + ((int64_t)b * p.R + r) * p.Lp + p.padl - p.A8 + l0, seg_bytes,
                      BAR(B_FULL + s));
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = ptx::idesc_f16(kM, kR2N, 0, 0);
    constexpr uint32_t descHiA = ptx::smem_desc_hi_sw128(1024);
    constexpr uint32_t descHiB = ((128u >> 4) & 0x3FFFu) | (1u << 14);      // SWIZZLE_NONE, 8-row groups 128 bytes apart
    for (int r = 0; r < p.R; ++r) {
      const int s = r % kD2Stages, ph = (r / kD2Stages) & 1;
      if (lane == 0) ptx::mbar_wait(BAR(B_FULL + s), ph);
      __syncwarp();
      ptx::tc_fence_after();
      if (ptx::elect_one()) {
        const uint32_t seg = STAGE(s) + nkk * Smem::kTile;
        for (int kst = 0; kst < p.nks; ++kst) {
          const int kk = kst >> 2, ks = kst & 3;
          const uint32_t alo = ptx::smem_desc_lo(STAGE(s) + kk * Smem::kTile, 16) + 2 * ks;
          const uint32_t blo = ptx::smem_desc_lo(seg + (uint32_t)(kst * 16) * 2, 16);
          ptx::mma_ss(tmem, ptx::make_desc(alo, descHiA), ptx::make_desc(blo, descHiB), idesc, (r | kst) ? 1u : 0u);
        }
        ptx::mma_commit(BAR(B_EMPTY + s));
        if (r == p.R - 1) ptx::mma_commit(BAR(B_ACC));
      }
      __syncwarp();
    }
  } else if (warp >= 4) {
    const int q4 = warp & 3, m = q4 * 32 + lane;                 // TMEM lane = (c_local, s)
    const uint32_t lane_addr = (uint32_t)(q4 * 32) << 16;
    const int c = cg * 16 + (m >> 3), sph = m & 7;
    const bool row_ok = c < p.C;
    ptx::mbar_wait(BAR(B_ACC), 0);
    ptx::tc_fence_after();
    const float sc = exp2f(-(float)(p.exps[0] + p.exps[1]));
    const float kap = *p.kappa, pscale = exp2f((float)p.exps[2]);
    const float* vrow = p.V + ((int64_t)b * p.C + (row_ok ? c : 0)) * p.L;
    __half* prow = p.P16out + ((int64_t)b * p.C + (row_ok ? c : 0)) * p.Lq;
    double acc = 0.0;
    // the 16 target values of chunk j + 1 are requested before chunk j is computed (one round trip per chunk, overlapped)
    float v[16], vn[16];
    auto load_v = [&](int j, float (&dst)[16]) {
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int l = l0 + 8 * (j * 16 + i) + sph;
        dst[i] = (row_ok && l < p.L) ? __ldg(vrow + l) : 0.f;
      }
    };
    load_v(0, vn);
#pragma unroll 1
    for (int j = 0; j < kR2N / 16; ++j) {
      uint32_t sr[16];
      ptx::tmem_ld16(tmem + lane_addr + j * 16, sr);
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = vn[i];
      if (j + 1 < kR2N / 16) load_v(j + 1, vn);
      ptx::tc_wait_ld();
      float a = 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int l = l0 + 8 * (j * 16 + i) + sph;
        const bool ok = row_ok && l < p.L;
        const float x = fmaf(__uint_as_float(sr[i]), sc, kEps);
        if (LOSS) {
          if (ok) a += v[i] * (__logf(v[i] + kEps) - __logf(x)) - v[i] + (x - kEps);         // metrics.py:22
        } else if (row_ok && l < p.Lq) {
          const float pv = ok ? fmaf(v[i], ptx::rcp_approx(x), -kap) * pscale : 0.f;         // nmf.py:65, centred
          prow[l] = __float2half_rn(fminf(pv, 65504.f));
        }
      }
      acc += (double)a;
    }
    if (LOSS) {
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (lane == 0) red[q4] = acc;
      asm volatile("bar.sync 1, 128;");
      if (q4 == 0 && lane == 0)
        p.loss_part[((int64_t)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x] = (red[0] + red[1]) + (red[2] + red[3]);
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem, kR2N);
}

// ---- operand preparation --------------------------------------------------------------------------------------------------
__device__ __forceinline__ int pow2_exp14(float mx) {
  if (!(mx > 0.f) || !isfinite(mx)) return 0;
  int e;
  frexpf(mx, &e);
  return 14 - e;
}

__global__ void __launch_bounds__(256)
absmax_kernel(const float* __restrict__ x, int64_t n, unsigned int* __restrict__ out) {
  float m = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) m = fmaxf(m, x[i]);
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(out, __float_as_uint(m));
}

// colsum[r] = sum over `outer` slabs of `inner` consecutive partials each: part[(o R + r) inner + i]; block r, fixed order.
// The block that finishes LAST also publishes kappa = sum(V) / sum_r colsum_W[r] colsum_H[r] (= sum of the reconstruction,
// nmf.py:776-779) and the exponent of the ratio tile (kappa 2^p in [2^-4, 2^-3)) when no other refresh follows in this call:
// two launches per refresh (prep, fold) instead of three.
struct FoldTail {
  const float* part;        // [(o R + r) inner + i]
  float* colsum;            // [R] of the factor being refreshed
  int outer, R, inner;
  unsigned int* ticket;     // zero between launches
  int do_kappa;
  const double* vsum;
  const float* colsum_all;  // [2 R]: W then H
  float* kappa;
  int* exps;
};

__global__ void __launch_bounds__(256)
fold_colsum_kernel(const FoldTail f) {
  __shared__ float sh[256];
  __shared__ bool is_last;
  const int r = blockIdx.x;
  const int64_t n = (int64_t)f.outer * f.inner;
  float a = 0.f;
  for (int64_t i = threadIdx.x; i < n; i += 256) {
    const int64_t o = i / f.inner, k = i - o * f.inner;
    a += f.part[(o * f.R + r) * f.inner + k];
  }
  sh[threadIdx.x] = a;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (threadIdx.x < w) sh[threadIdx.x] += sh[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    f.colsum[r] = sh[0];
    __threadfence();                                            // this component's sum is visible before the ticket is
    is_last = atomicAdd(f.ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!is_last || threadIdx.x != 0) return;
  __threadfence();
  *f.ticket = 0u;
  if (f.do_kappa) {
    double dot = 0.0;
    for (int q = 0; q < f.R; ++q) dot += (double)__ldcg(f.colsum_all + q) * (double)__ldcg(f.colsum_all + f.R + q);
    const float k = (float)(*f.vsum / dot);
    int e = 0;
    const bool ok = k > 0.f && isfinite(k);
    if (ok) { frexpf(k, &e); e = -3 - e; }
    *f.kappa = ok ? k : 0.f;
    f.exps[2] = e;
  }
}

// One pass over W (C, R, T), block c: both fp16 operand copies of this row, scaled by 2^eW (eW from the max of W), written
// 16 bytes per thread and step, plus the row's per-component sums (-> colsum_W, nmf.py:128-131):
//   Ws16[(c, grp, r%16, s)][u]   = W[c, r, u - s]              (dgrad, eight shifted copies)
//   Wsh16[(c, s)][r Tq + u]      = W[c, r, s + A8 - u]         (recon, eight shifted copies)
//
// The eight shifted copies dominate (cfg3: 100 MB per refresh).  Every 16-byte store gathers eight CONSECUTIVE shifts of one
// component, so the lanes of a warp read W at addresses eight floats apart: from a dense shared-memory row that is an 8-way
// bank conflict per load, and with per-element index arithmetic and bounds checks the kernel was instruction-bound on top
// (36 us at cfg3, 2.8 TB/s).  Hence the row is staged scaled and DE-INTERLEAVED by shift residue:
//     stage[r][t & 7][(t >> 3) + F]   for t in [-8 F, 8 (S - F)),  zero outside [0, T)
// (S slots per residue class, F leading ones).  For a fixed copy index s (an unrolled loop) element k of a store then
// sits at a compile-time class and a compile-time slot offset from the thread's base, consecutive lanes read consecutive
// words, and out-of-range shifts read the zero margins: eight loads with immediate offsets, four packs, one store.  Stores
// whose eight shifts all fall outside [0, T) are skipped: those bytes are zero from tc_nmfd_create on and nobody writes them.
__device__ __forceinline__ void prep_w_shifted(const float* __restrict__ stage, int S, int F, int R, int T, int Tq, int A8,
                                               int ngroups, int c, __half* __restrict__ Ws16, __half* __restrict__ Wsh16) {
  const int NV = Tq >> 3;                                  // 16-byte stores per row of either copy
  const unsigned int magic = 0xFFFFFFFFu / (unsigned)NV + 1u;     // j / NV == umulhi(j, magic) for the j below (< 2^16)
  const int64_t rows = (int64_t)ngroups * 128;
  auto pack8 = [](const float (&v)[8]) {
    __half2 h[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
    return *reinterpret_cast<const uint4*>(h);
  };
  // one item = one (component r, 8-shift group vec): its eight stores (the eight copies of one layout) share every address
  // computation; inside, copy index and element index are compile-time, so a load is [base + class S + immediate].
  // dgrad copies: Ws16[(c, grp, r % 16, SH)][u + k] = W[c, r, u + k - SH]
  for (int j = threadIdx.x; j < R * NV; j += 256) {
    const int r = (int)__umulhi((unsigned)j, magic), vec = j - r * NV, u = vec << 3;
    const float* up = stage + (int64_t)r * 8 * S + F + vec;                     // ascending windows
    __half* ws = Ws16 + ((int64_t)c * rows + (int64_t)(r >> 4) * 128 + (r & 15) * 8) * Tq + u;       // + SH Tq
#pragma unroll
    for (int SH = 0; SH < 8; ++SH) {
      if (u + 7 - SH >= 0 && u - SH < T) {
        float v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = up[((k - SH) & 7) * S + ((k - SH) >> 3)];
        *reinterpret_cast<uint4*>(ws + SH * Tq) = pack8(v);
      }
    }
  }
  // recon copies: Wsh16[(c, SH)][r Tq + u + k] = W[c, r, SH + A8 - u - k]
  const int64_t wsh_step = (int64_t)R * Tq;
  for (int j = threadIdx.x; j < R * NV; j += 256) {
    const int r = (int)__umulhi((unsigned)j, magic), vec = j - r * NV, u = vec << 3;
    const float* dn = stage + (int64_t)r * 8 * S + F + (A8 >> 3) - vec;         // descending windows
    __half* wsh = Wsh16 + (int64_t)c * 8 * wsh_step + (int64_t)r * Tq + u;      // + SH R Tq
#pragma unroll
    for (int SH = 0; SH < 8; ++SH) {
      if (SH + A8 - u >= 0 && SH + A8 - u - 7 < T) {
        float v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = dn[((SH - k) & 7) * S + ((SH - k) >> 3)];
        *reinterpret_cast<uint4*>(wsh + SH * wsh_step) = pack8(v);
      }
    }
  }
}

__global__ void __launch_bounds__(256, 8)     // 8 blocks per SM: the 1025 blocks of cfg3 run as one wave
prep_w_kernel(const float* __restrict__ W, int C, int R, int T, int Tq, int ngroups,
              const unsigned int* __restrict__ absmax, int* __restrict__ exps, __half* __restrict__ Ws16,
              __half* __restrict__ Wsh16, int A8, float* __restrict__ cs_part, int use_smem, int S, int F) {
  const int e = pow2_exp14(__uint_as_float(*absmax));
  if (blockIdx.x == 0 && threadIdx.x == 0) exps[0] = e;
  const float sc = exp2f((float)e);
  const int c = blockIdx.x;
  const float* Wg = W + (int64_t)c * R * T;
  extern __shared__ float stage[];
  auto w_at = [&](int r, int t) { return (r < R && t >= 0 && t < T) ? Wg[r * T + t] * sc : 0.f; };
  auto pack8 = [&](const float (&v)[8]) {
    __half2 h[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
    return *reinterpret_cast<const uint4*>(h);
  };
  if (use_smem) {
    for (int i = threadIdx.x; i < R * 8 * S; i += 256) stage[i] = 0.f;
    __syncthreads();
    // the row's R T values: eight independent loads in flight per thread before the first dependent shared-memory store
    // (a loop of load -> store pairs paid the full memory latency R times per block and was what bounded this kernel)
    const int RT = R * T;
    const unsigned int magic_t = 0xFFFFFFFFu / (unsigned)T + 1u;          // i / T == umulhi(i, magic_t): R T < 2^16 here
    for (int i0 = threadIdx.x; i0 < RT; i0 += 256 * 8) {
      float x[8];
#pragma unroll
      for (int m = 0; m < 8; ++m) { const int i = i0 + m * 256; x[m] = i < RT ? Wg[i] : 0.f; }
#pragma unroll
      for (int m = 0; m < 8; ++m) {
        const int i = i0 + m * 256;
        if (i < RT) {
          const int r = (int)__umulhi((unsigned)i, magic_t), t = i - r * T;
          stage[(r * 8 + (t & 7)) * S + (t >> 3) + F] = x[m] * sc;
        }
      }
    }
    __syncthreads();
    prep_w_shifted(stage, S, F, R, T, Tq, A8, ngroups, c, Ws16, Wsh16);
  } else {                           // a row of W too long to stage: straight from global memory, every store written
    const int64_t rows = (int64_t)ngroups * 128;
    for (int i8 = threadIdx.x; i8 < rows * Tq / 8; i8 += 256) {
      const int i = i8 * 8, n = i / Tq, u = i - n * Tq;
      const int r = (n >> 7) * 16 + ((n & 127) >> 3), sh = n & 7;
      float v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = w_at(r, u + k - sh);
      *reinterpret_cast<uint4*>(Ws16 + ((int64_t)c * rows + n) * Tq + u) = pack8(v);
    }
    for (int i8 = threadIdx.x; i8 < 8 * R * Tq / 8; i8 += 256) {
      const int i = i8 * 8, sh = i / (R * Tq), ru = i - sh * (R * Tq), r = ru / Tq, u = ru - r * Tq;
      float v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = w_at(r, sh + A8 - u - k);
      *reinterpret_cast<uint4*>(Wsh16 + ((int64_t)c * 8 + sh) * ((int64_t)R * Tq) + ru) = pack8(v);
    }
  }
  // per-component sums of this row: warp w takes r = w, w + 8, ...; fixed order
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int r = warp; r < R; r += 8) {
    float a = 0.f;
    for (int t = lane; t < T; t += 32) a += Wg[r * T + t];
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) cs_part[(int64_t)c * R + r] = a;
  }
}

// H (B, R, Lin) fp32 -> Hp16 (B R rows x Lp): H[b,r,j] 2^eH at column padl + j (margins stay zero), 2048 elements per
// block, + the block's partial sum (-> colsum_H, nmf.py:122-125).  grid (chunks, B R)
__global__ void __launch_bounds__(256)
prep_h_kernel(const float* __restrict__ H, int Lin, int Lp, int padl, const unsigned int* __restrict__ absmax,
              int* __restrict__ exps, __half* __restrict__ Hp16, float* __restrict__ cs_part) {
  __shared__ float sh[8];
  const int e = pow2_exp14(__uint_as_float(*absmax));
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) exps[1] = e;
  const float sc = exp2f((float)e);
  const int64_t row = blockIdx.y;
  const int j = blockIdx.x * 2048 + threadIdx.x * 8;
  float a = 0.f;
  if (j < Lin) {
    float v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) { v[k] = j + k < Lin ? H[row * Lin + j + k] : 0.f; a += v[k]; v[k] *= sc; }
    __half2 h[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
    *reinterpret_cast<uint4*>(Hp16 + row * Lp + padl + j) = *reinterpret_cast<const uint4*>(h);
  }
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += sh[i];
    cs_part[row * gridDim.x + blockIdx.x] = t;
  }
}

__global__ void __launch_bounds__(256)
vsum_kernel(const float* __restrict__ V, int64_t n, double* __restrict__ part) {
  __shared__ double sh[8];
  double a = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) a += (double)V[i];
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x == 0) { double t = 0.0; for (int i = 0; i < 8; ++i) t += sh[i]; part[blockIdx.x] = t; }
}

// Dynamic shared memory of each launch (bytes; the tcgen05 kernels' counts include 1 KB for aligning their base to 1024).
// The recon2 / dgrad2 stages are the layouts computed at the top of those kernels; prep_w_kernel stages a row of W when it
// fits (its division by multiplication also needs R T < 2^16) and reads it from global memory otherwise (0 bytes).
struct KernelSmem {
  int recon2, dgrad2, wgrad, prep_w;
};

KernelSmem kernel_smem(const NmfdShape& d, int Tq, int S) {
  KernelSmem k;
  const int nkk = Tq / kKB;
  const uint32_t st_r = (((uint32_t)nkk * Smem::kTile + (uint32_t)(8 * kR2N + Tq) * 2) + 1023u) & ~1023u;
  k.recon2 = (int)(kD2Stages * st_r + 8 * (2 * kD2Stages + 1) + 16 + 64 + 1024);
  const uint32_t seg_pitch = (((uint32_t)(1024 + Tq) * 2) + 127u) & ~127u;
  const uint32_t st_d = (((uint32_t)nkk * Smem::kTile + kD2Q * seg_pitch) + 1023u) & ~1023u;
  k.dgrad2 = (int)(kD2Stages * st_d + 8 * (2 * kD2Stages + 1) + 16 + 1024);
  k.wgrad = Smem::kTotal + 1024;
  const size_t wrow_bytes = (size_t)d.R * 8 * S * sizeof(float);
  k.prep_w = (wrow_bytes <= 200 * 1024 && (int64_t)d.R * d.T < 65536) ? (int)wrow_bytes : 0;
  return k;
}

// The limit is per kernel and per device, and other contexts on this device may need more than this one: only raise it.
template <class Kernel>
int raise_smem_limit(Kernel* kern, int bytes) {
  cudaFuncAttributes fa;
  NMF_CUDA_CHECK(cudaFuncGetAttributes(&fa, kern));
  if (fa.maxDynamicSharedSizeBytes < bytes)
    NMF_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  return 0;
}

}  // namespace

struct TcNmfdState {
  NmfdShape d{};
  int Lp = 0, padl = 0, Lq = 0, Cpad = 0;
  __half *Hp16 = nullptr, *P16 = nullptr, *Ws16 = nullptr, *Wsh16 = nullptr;
  int A8 = 0;                       // T - 1 rounded up to 8: alignment of the H window of the eight-phase recon
  int Tq = 0, ngroups = 1, cps_h2 = 0, ws_h2 = 1;   // dgrad2: padded shift extent, 16-component groups, c per split, splits
  int ws_w = 1, kbs_w = 0;          // wgrad: splits, k-blocks per split
  int prep_S = 0, prep_F = 0;       // staging layout of prep_w_kernel: S slots per shift-residue class, F leading zeros
  KernelSmem smem{};
  float* part = nullptr;            // wgrad / dgrad split partials
  int64_t part_floats = 0;
  unsigned int* absmax = nullptr;   // [2]: max of W, max of H (float bits; written by absmax_kernel or by the ratio stage)
  float* colsum = nullptr;          // [2][R]: colsum_W | colsum_H
  float* cs_part = nullptr;         // per-row / per-block partial sums of the factor being refreshed
  bool w_fresh = false, h_fresh = false;      // the fp16 copies / column sums of W, H match the fp32 factor
  bool aw_valid = false, ah_valid = false;    // absmax[0], absmax[1] hold the max of the current W, H
  int* exps = nullptr;              // {eW, eH, eP}
  float* kappa = nullptr;
  double* vsum = nullptr;           // [1] + [256] partials
  double* loss_part = nullptr;
  int loss_blocks = 0;
  CUtensorMap tmP, tmWs, tmWsh;
};

bool tc_nmfd_shape_supported(const NmfdShape& d) {
  return d.one_d() && d.T >= 1 && d.T <= 128 && d.R >= 1 && d.R <= 256;
}

void tc_nmfd_destroy(TcNmfdState* s) {
  if (!s) return;
  cudaFree(s->Wsh16); cudaFree(s->Ws16); cudaFree(s->Hp16); cudaFree(s->P16); cudaFree(s->part); cudaFree(s->absmax);
  cudaFree(s->colsum); cudaFree(s->cs_part); cudaFree(s->exps); cudaFree(s->kappa); cudaFree(s->vsum); cudaFree(s->loss_part);
  delete s;
}

int tc_nmfd_create(TcNmfdState** out, const NmfdShape& d) {
  *out = nullptr;
  TcNmfdState* s = new TcNmfdState();
  s->d = d;
  const int Tp = (int)round_up(d.T, kKB);
  s->padl = (int)round_up(Tp + 136, 8);                          // every window start >= 0 (padl >= A8 as well)
  s->Lp = (int)round_up((int64_t)s->padl + round_up((int64_t)d.L, 8 * kR2N) + 256 + kWinHalfs + 136, 8);
  s->A8 = (int)round_up(d.T - 1, 8);
  s->Tq = (int)round_up(s->A8 + 8, kKB);                            // shifts u in [0, A8 + 7]; also covers dgrad's [0, T + 6]
  s->ngroups = (int)ceil_div(d.R, 16);
  s->Lq = (int)round_up(round_up((int64_t)d.L, 2048) + 1024 + s->Tq + kWinHalfs + 8, 8);
  s->Cpad = (int)round_up(d.C, kM);
  // split the K loops of wgrad / dgrad so that the grid is a few waves of 148 CTAs
  const int64_t tiles_w = ceil_div(d.C, kM) * d.R, kb_w = (int64_t)d.B * ceil_div(d.L, kKB);
  s->ws_w = (int)std::max<int64_t>(1, std::min<int64_t>(kb_w / 8, ceil_div(148 * 4, tiles_w)));
  s->kbs_w = (int)ceil_div(kb_w, s->ws_w); s->ws_w = (int)ceil_div(kb_w, s->kbs_w);
  {
    const int64_t tiles = ceil_div(d.Lin, kD2Q * 1024) * d.B * s->ngroups;
    int64_t ws = std::max<int64_t>(1, std::min<int64_t>(d.C / 4 > 0 ? d.C / 4 : 1, ceil_div(148, tiles)));
    s->cps_h2 = (int)ceil_div(d.C, ws);
    s->ws_h2 = (int)ceil_div(d.C, s->cps_h2);
  }
  // staging layout of prep_w_kernel: shifts down to A8 + 1 - Tq
  s->prep_F = (s->Tq - s->A8) / 8 + 2;
  s->prep_S = s->Tq / 8 + s->prep_F;
  s->smem = kernel_smem(d, s->Tq, s->prep_S);
  const KernelSmem& k = s->smem;
  if (std::max(std::max(k.recon2, k.dgrad2), std::max(k.wgrad, k.prep_w)) > 232448) {
    delete s;
    set_error("internal: tc_nmfd_create: the shared-memory stages exceed 227 KB for T = " + std::to_string(d.T));
    return -1;
  }
  int rc = 0;
  if (!rc) rc = raise_smem_limit(tcnmfd_recon2_kernel<false>, k.recon2);
  if (!rc) rc = raise_smem_limit(tcnmfd_recon2_kernel<true>, k.recon2);
  if (!rc) rc = raise_smem_limit(tcnmfd_dgrad2_kernel, k.dgrad2);
  if (!rc) rc = raise_smem_limit(tcnmfd_wgrad_kernel, k.wgrad);
  if (!rc) rc = raise_smem_limit(prep_w_kernel, k.prep_w);
  if (rc) { delete s; return rc; }
  const int64_t pw = (int64_t)s->ws_w * d.C * d.R * d.T, ph = (int64_t)s->ws_h2 * d.B * d.R * d.Lin;
  s->part_floats = pw > ph ? pw : ph;
  s->loss_blocks = (int)(ceil_div(d.L, 8 * kR2N) * ceil_div(d.C, 16) * d.B);
  const size_t hbytes = (size_t)d.B * d.R * s->Lp * 2;
  const size_t pbytes = ((size_t)d.B * d.C + 1) * s->Lq * 2;
  cudaError_t e = cudaSuccess;
  const size_t wshbytes = (size_t)s->Cpad * 8 * d.R * s->Tq * 2;
  if (e == cudaSuccess) e = cudaMalloc(&s->Wsh16, wshbytes);
  if (e == cudaSuccess) e = cudaMemset(s->Wsh16, 0, wshbytes);
  const size_t wsbytes = (size_t)s->Cpad * s->ngroups * 128 * s->Tq * 2;
  if (e == cudaSuccess) e = cudaMalloc(&s->Ws16, wsbytes);
  if (e == cudaSuccess) e = cudaMemset(s->Ws16, 0, wsbytes);
  if (e == cudaSuccess) e = cudaMalloc(&s->Hp16, hbytes);
  if (e == cudaSuccess) e = cudaMalloc(&s->P16, pbytes);
  if (e == cudaSuccess) e = cudaMalloc(&s->part, (size_t)s->part_floats * 4);
  if (e == cudaSuccess) e = cudaMalloc(&s->absmax, 2 * sizeof(unsigned int));
  if (e == cudaSuccess) e = cudaMalloc(&s->colsum, 2 * (size_t)d.R * sizeof(float));
  {
    const int64_t np = std::max<int64_t>((int64_t)d.C * d.R, (int64_t)d.B * d.R * ceil_div(d.Lin, 2048));
    if (e == cudaSuccess) e = cudaMalloc(&s->cs_part, (size_t)np * sizeof(float));
  }
  if (e == cudaSuccess) e = cudaMalloc(&s->exps, 8 * sizeof(int));          // [0..3] exponents, [4..5] fold tickets
  if (e == cudaSuccess) e = cudaMemset(s->exps, 0, 8 * sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc(&s->kappa, sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&s->vsum, 257 * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&s->loss_part, (size_t)s->loss_blocks * sizeof(double));
  if (e == cudaSuccess) e = cudaMemset(s->Hp16, 0, hbytes);
  if (e == cudaSuccess) e = cudaMemset(s->P16, 0, pbytes);
  if (e == cudaSuccess) e = cudaMemset(s->exps, 0, 4 * sizeof(int));
  if (e != cudaSuccess) {
    tc_nmfd_destroy(s);
    set_error(std::string("tc_nmfd_create: ") + cudaGetErrorString(e));
    return 2;
  }
  rc |= make_tmap(&s->tmP, s->P16, (int64_t)d.B * d.C, s->Lq, s->Lq, kM);
  rc |= make_tmap(&s->tmWs, s->Ws16, (int64_t)s->Cpad * s->ngroups * 128, s->Tq, s->Tq, 128);
  rc |= make_tmap(&s->tmWsh, s->Wsh16, (int64_t)s->Cpad * 8, (int64_t)d.R * s->Tq, (int64_t)d.R * s->Tq, 128);
  if (rc) { tc_nmfd_destroy(s); return 2; }
  *out = s;
  return 0;
}

int tc_nmfd_set_target(TcNmfdState* s, const float* V, double* vsum_host, cudaStream_t st) {
  const int64_t n = (int64_t)s->d.B * s->d.C * s->d.L;
  vsum_kernel<<<256, 256, 0, st>>>(V, n, s->vsum + 1);
  NMF_LAUNCH_CHECK();
  int rc = sum_partials(s->vsum + 1, 256, s->vsum, st);
  if (rc) return rc;
  NMF_CUDA_CHECK(cudaMemcpyAsync(vsum_host, s->vsum, sizeof(double), cudaMemcpyDeviceToHost, st));
  NMF_CUDA_CHECK(cudaStreamSynchronize(st));
  return 0;
}

namespace {

// arguments of the fold launch after a preparation launch: fold `outer x R x inner` partial sums into colsum[which], then kappa if this is the
// last refresh of the call
FoldTail fold_tail_args(TcNmfdState* s, int which, int outer, int inner, int do_kappa) {
  FoldTail f{};
  f.part = s->cs_part; f.colsum = s->colsum + (which ? s->d.R : 0); f.outer = outer; f.R = s->d.R; f.inner = inner;
  f.ticket = reinterpret_cast<unsigned int*>(s->exps + 4 + which); f.do_kappa = do_kappa;
  f.vsum = s->vsum; f.colsum_all = s->colsum; f.kappa = s->kappa; f.exps = s->exps;
  return f;
}

// bring the fp16 operand copies, column sums (and with them kappa) up to date with the fp32 factors: only what changed
int refresh(TcNmfdState* s, const float* W, const float* H, cudaStream_t st) {
  const NmfdShape& d = s->d;
  if (!s->w_fresh) {
    if (!s->aw_valid) {
      NMF_CUDA_CHECK(cudaMemsetAsync(s->absmax, 0, sizeof(unsigned int), st));
      absmax_kernel<<<256, 256, 0, st>>>(W, (int64_t)d.C * d.R * d.T, s->absmax);
      NMF_LAUNCH_CHECK();
      s->aw_valid = true;
    }
    prep_w_kernel<<<d.C, 256, s->smem.prep_w, st>>>(W, d.C, d.R, d.T, s->Tq, s->ngroups, s->absmax, s->exps, s->Ws16,
                                                    s->Wsh16, s->A8, s->cs_part, s->smem.prep_w > 0 ? 1 : 0, s->prep_S,
                                                    s->prep_F);
    NMF_LAUNCH_CHECK();
    fold_colsum_kernel<<<d.R, 256, 0, st>>>(fold_tail_args(s, 0, d.C, 1, /*do_kappa=*/s->h_fresh));
    NMF_LAUNCH_CHECK();
    s->w_fresh = true;
  }
  if (!s->h_fresh) {
    if (!s->ah_valid) {
      NMF_CUDA_CHECK(cudaMemsetAsync(s->absmax + 1, 0, sizeof(unsigned int), st));
      absmax_kernel<<<256, 256, 0, st>>>(H, (int64_t)d.B * d.R * d.Lin, s->absmax + 1);
      NMF_LAUNCH_CHECK();
      s->ah_valid = true;
    }
    const int nch = (int)ceil_div(d.Lin, 2048);
    dim3 gh((unsigned)nch, (unsigned)(d.B * d.R));
    prep_h_kernel<<<gh, 256, 0, st>>>(H, d.Lin, s->Lp, s->padl, s->absmax + 1, s->exps, s->Hp16, s->cs_part);
    NMF_LAUNCH_CHECK();
    fold_colsum_kernel<<<d.R, 256, 0, st>>>(fold_tail_args(s, 1, d.B, nch, /*do_kappa=*/1));
    NMF_LAUNCH_CHECK();
    s->h_fresh = true;
  }
  return 0;
}

}  // namespace

int tc_nmfd_recon(TcNmfdState* s, const float* V, const float* W, const float* H, bool loss, double* loss_dev,
                  cudaStream_t st) {
  int rc = refresh(s, W, H, st);
  if (rc) return rc;
  const NmfdShape& d = s->d;
  Recon2Params q{};
  q.B = d.B; q.C = d.C; q.L = d.L; q.R = d.R; q.Lp = s->Lp; q.padl = s->padl; q.Lq = s->Lq; q.Tq = s->Tq; q.A8 = s->A8;
  q.nks = (int)ceil_div(s->A8 + 8, 16);
  q.Hp16 = s->Hp16; q.P16out = s->P16; q.V = V; q.exps = s->exps; q.kappa = s->kappa; q.loss_part = s->loss_part;
  dim3 grid((unsigned)ceil_div(d.L, 8 * kR2N), (unsigned)ceil_div(d.C, 16), (unsigned)d.B);
  if (loss) {
    tcnmfd_recon2_kernel<true><<<grid, kD2Threads, s->smem.recon2, st>>>(s->tmWsh, q);
    NMF_LAUNCH_CHECK();
    return sum_partials(s->loss_part, (int)(grid.x * grid.y * grid.z), loss_dev, st);
  }
  tcnmfd_recon2_kernel<false><<<grid, kD2Threads, s->smem.recon2, st>>>(s->tmWsh, q);
  NMF_LAUNCH_CHECK();
  return 0;
}

// numerator partials of the W update from the P16 written by the last recon: [*nsplit][C][R][T] fp32
int tc_nmfd_wgrad(TcNmfdState* s, const float** part, int* nsplit, cudaStream_t st) {
  const NmfdShape& d = s->d;
  WgradParams p{};
  p.B = d.B; p.C = d.C; p.L = d.L; p.R = d.R; p.T = d.T; p.Lp = s->Lp; p.padl = s->padl;
  p.Hp16 = s->Hp16; p.exps = s->exps; p.out = s->part; p.kb_per_split = s->kbs_w;
  dim3 grid((unsigned)ceil_div(d.C, kM), (unsigned)d.R, (unsigned)s->ws_w);
  tcnmfd_wgrad_kernel<<<grid, kThreads, s->smem.wgrad, st>>>(s->tmP, p);
  NMF_LAUNCH_CHECK();
  *part = s->part; *nsplit = s->ws_w;
  return 0;
}

int tc_nmfd_dgrad(TcNmfdState* s, const float** part, int* nsplit, cudaStream_t st) {
  const NmfdShape& d = s->d;
  Dgrad2Params q{};
  q.B = d.B; q.C = d.C; q.R = d.R; q.Lin = d.Lin; q.Lq = s->Lq; q.Tq = s->Tq; q.ngroups = s->ngroups;
  q.P16 = s->P16; q.exps = s->exps; q.out = s->part; q.c_per_split = s->cps_h2;
  q.nks = (int)ceil_div(d.T + 7, 16);
  dim3 grid((unsigned)ceil_div(d.Lin, kD2Q * 1024), (unsigned)s->ws_h2, (unsigned)(d.B * s->ngroups));
  tcnmfd_dgrad2_kernel<<<grid, kD2Threads, s->smem.dgrad2, st>>>(s->tmWs, q);
  NMF_LAUNCH_CHECK();
  *part = s->part; *nsplit = s->ws_h2;
  return 0;
}

const float* tc_nmfd_kappa(const TcNmfdState* s) { return s->kappa; }
const float* tc_nmfd_colsum(const TcNmfdState* s) { return s->colsum; }

// The caller is about to overwrite a factor (which = 0: W, 1: H) with its ratio stage: returns the slot the stage should
// atomicMax the new values into (zeroed here), so the next refresh needs no separate pass for the operand exponent.
unsigned int* tc_nmfd_begin_update(TcNmfdState* s, int which, cudaStream_t st) {
  unsigned int* slot = s->absmax + which;
  if (cudaMemsetAsync(slot, 0, sizeof(unsigned int), st) != cudaSuccess) return nullptr;
  if (which == 0) { s->w_fresh = false; s->aw_valid = true; } else { s->h_fresh = false; s->ah_valid = true; }
  return slot;
}

// a factor was changed by someone else: everything derived from it is stale
void tc_nmfd_mark_dirty(TcNmfdState* s) {
  s->w_fresh = s->h_fresh = false;
  s->aw_valid = s->ah_valid = false;
}

int tc_nmfd_check_wait_abort() { return ptx::check_wait_abort("NMFD "); }

}  // namespace nmfb200
