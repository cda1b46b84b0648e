// Tensor-core path of the dense NMF factor update for sm_100a: tcgen05.mma + TMEM + TMA.
//
// One persistent, warp-specialised CTA per SM walks work items (128-row block of the row factor F,
// chunk of 128-column tiles).  Per tile (FlashAttention-shaped, but with a ratio instead of softmax):
//
//   TMA      G tile [128 c][KW] and V tile [128 m][128 c] (fp16, SWIZZLE_128B) -> shared memory
//   MMA-1    S[128 m][128 c]  = F_blk G_tile^T            tcgen05.mma SS, fp32 accumulators in TMEM
//   ratio    P = V * rcp(S*c1 + c2)  (== V / (F G^T + eps), nmf.py:65); the CENTRED tile P - kappa -> fp16, written
//            back to TMEM over S columns the writer has already read (256 threads per tile: two warpgroups, each all 128
//            TMEM lanes x half the columns)
//   MMA-2    O[128 m][KW]   += (P - kappa) G_tile          tcgen05.mma TS (A from TMEM, B = G tile MN-major)
//            (numerator = O + kappa colsum(G), added in fp32 by the ratio stage)
//
// so neither S = WH nor P = V/(WH) ever leaves the SM (nmf.py:376-378 materialises both in HBM).
// F/G are fp16 copies of the factors scaled by a power of two; in split mode they carry hi|lo halves
// (KW = 2*Rp) and S = Fhi Ghi + Flo Ghi + Fhi Glo, O = P [Ghi|Glo] recovers ~22-bit factors.
//
// Warp roles (512 threads): 0-3, 4-7 ratio warpgroups (left / right half of the tile's columns) | 8-11 epilogue (O -> fp32
// partial numerators) | 12 TMA producer for V (the HBM stream, own ring) | 13 MMA issuer for S (one lane) | 14 TMA producer
// for F/G (L2-resident factors) | 15 MMA issuer for O.  The control warps have the highest ids = highest issue priority.
// S runs up to NS tiles ahead of O in the tensor pipe, across work-item boundaries.
#include "tc_nmf.cuh"

#include <cooperative_groups.h>
#include <cuda.h>
#include <cudaTypedefs.h>

#include <cstdlib>
#include <cstring>
#include <string>

#include "sm100_ptx.cuh"

namespace nmfb200 {

namespace {

constexpr int kTileM = 128;          // rows of the row factor per work item (= TMEM lanes)
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kColS = 0;        // S/P stages: columns [TN i, TN i + TN); O accumulator follows at NS * TN

// Compile-time configuration of the fused kernel.
//   RP    padded rank (64 or 128);  SPLIT  hi|lo fp16 factors (KW = 2 RP operand columns)
//   TN    tile width in columns of V (64 or 128): narrower tiles = deeper rings in the same shared memory
//   NF / NG / NV  F blocks, G-tile ring, V-tile ring;  NS  S/P accumulator stages in TMEM (the S-MMA warp runs up to
//   NS tiles ahead of the O-MMA warp)
//   NRW   ratio warpgroups (each processes TN / NRW columns of every tile)
// The ratio tile P is written over the S columns of its stage; the stage is free again when the O-MMA has consumed P.
constexpr unsigned kEpiPaceNs = 100;     // pause between the epilogue's row stores (see the epilogue warpgroup)

template <int RP_, bool SPLIT_, int TN_, int NF_, int NG_, int NV_, int NS_, int NRW_ = 2>
struct Cfg {
  static constexpr int RP = RP_, TN = TN_, NF = NF_, NG = NG_, NV = NV_, NS = NS_, NRW = NRW_;
  // 4 NRW ratio warps, then 4 epilogue warps, then 4 control warps (TMA V / MMA S / TMA F,G / MMA O)
  static constexpr int kThreads = 128 + 128 * NRW_ + 128;
  static constexpr bool SPLIT = SPLIT_;
  static constexpr int KW = RP_ * (SPLIT_ ? 2 : 1);
};

struct TcKernelParams {
  int Mr, Nc;                 // valid rows of F / rows of G (= columns of Vm)
  int row_blocks, tiles, nchunks, tiles_per_chunk;
  float* part;                // [nchunks][Mr][ldp] fp32 numerators
  float* part2;               // [nchunks][Mr][ldp] fp32 denominators (beta != 1 kernels)
  float bm1, bm2;             // beta - 1, beta - 2 (generic-beta kernel)
  int64_t chunk_stride;
  int ldp;
  const int* exps;            // device: {v, aW, aH, p, pn, pd}: power-of-two exponents of V16, W16, H16, of the KL ratio
                              // tile P, and of the two beta != 1 tiles Pn, Pp
  int ef, eg;                 // which of exps[] belong to F and G
  double* loss_part;          // LOSS mode: [gridDim.x][2] = {sum v~ lg2(x), sum S~}
  const float* kappa;         // device scalar: centring constant of the ratio tile (typical P), 0 = off
};

// shared memory: NF F blocks | NG G-tile ring | NV V-tile ring | mbarriers | tmem ptr | loss slots
template <int KW, int TN, int NF, int NG, int NV, int NS>
struct SmemLayout {
  static constexpr int kFBytes = kTileM * KW * 2;
  static constexpr int kGBytes = TN * KW * 2;
  static constexpr int kVBytes = kTileM * TN * 2;
  static constexpr int kF = 0;
  static constexpr int kG = kF + NF * kFBytes;
  static constexpr int kV = kG + NG * kGBytes;
  static constexpr int kBar = kV + NV * kVBytes;
  static constexpr int kNumBars = 2 * NF + 2 * NG + 2 * NV + 3 * NS + 2;
  static constexpr int kTmemPtr = (kBar + 8 * kNumBars + 15) / 16 * 16;   // loss slots 16-byte aligned: paired doubles
  static constexpr int kLossSlots = kTmemPtr + 16;
  static constexpr int kTotal = kLossSlots + 16 * 16;
};

// BM selects the phi stage (nmf.py:61-74): 0 = beta 1 (one centred ratio tile, one accumulator); otherwise two tiles
// Pn = V x^(beta-2), Pp = x^(beta-1) and two accumulators (numerator, denominator): 1 = beta 0, 2 = beta 0.5,
// 3 = beta 1.5, 4 = any other beta (lg2/ex2).
// 5 = beta 2: the tile is the scale-matched residual V - kappa WH (signed, no MUFU work); numerator = O + kappa W (H^T H)
// is rebuilt in fp32 by the ratio stage, the same trick as the kappa centring of beta 1 (all-positive sums would inherit the
// tensor cores' truncation bias).
enum : int { kBmKL = 0, kBmIS = 1, kBm05 = 2, kBm15 = 3, kBmGen = 4, kBmEU = 5 };

// FOLD (beta 1 update kernels only): the W update's contraction ALSO accumulates the loss sums of the LOSS kernel from the S
// tile it forms anyway (metrics.py:22 needs sum V lg(WH + eps) and sum WH at exactly the factors the next W update starts
// from), so the loss evaluation of every 10th iteration costs one lg2 per element instead of a pass over V of its own.
template <class C, int BM, bool LOSS, bool FOLD = false>
__global__ void __launch_bounds__(C::kThreads, 1)
tc_contract_kernel(const __grid_constant__ CUtensorMap tmF, const __grid_constant__ CUtensorMap tmG,
                   const __grid_constant__ CUtensorMap tmV, const TcKernelParams p) {
  constexpr int RP = C::RP, KW = C::KW, TN = C::TN, NF = C::NF, NG = C::NG, NV = C::NV, NS = C::NS;
  constexpr bool SPLIT = C::SPLIT;
  constexpr int NRW = C::NRW;
  // Warp roles by warp id.  The warp scheduler of an SM sub-partition prefers the HIGHEST warp id among its eligible warps
  // (B300_MICROARCH.md, "arbiter priority: hi-wid-first"), and the TMA producers / MMA issuers are short serial
  // instruction streams on the critical path of every tile hand-off: they get the top four ids (one per sub-partition),
  // the throughput-bound ratio warps the lowest.  (Round 1 had them at ids 0-3: a wake-up of an issuing warp took 500-900
  // cycles while the ratio warps of its sub-partition were busy, profiles/r2_trace_*.txt.)
  constexpr int kEpiWarp0 = 4 * NRW;              // first epilogue warp (ratio warps are 0 .. 4 NRW - 1)
  constexpr int kCtl0 = 4 * NRW + 4;              // control warps: +0 TMA (V) | +1 MMA issuer S | +2 TMA (F, G) | +3 MMA issuer O
  constexpr bool TWO = BM != kBmKL && BM != kBmEU && !LOSS;     // LOSS kernels only need S, whatever the beta
  constexpr bool EU = BM == kBmEU;
  // TMEM columns.  one-output: S/P stages [0, NS TN) | O [NS TN, NS TN + KW).
  //               two-output: S/Pn stages [0, 256) | Pp stages [256, 384) | O_num [384, 448) | O_den [448, 512)
  constexpr uint32_t kColPp = NS * TN;
  constexpr uint32_t kColO = TWO ? 384 : NS * TN;
  constexpr uint32_t kColO2 = 448;
  using L = SmemLayout<KW, TN, NF, NG, NV, NS>;
  static_assert(TWO || (int)kColO + KW <= (int)kTmemCols, "TMEM budget");
  static_assert(!TWO || (!SPLIT && RP == 64 && TN == 128 && NS == 2), "two-output kernels: fast mode, R <= 64");
  static_assert(TN == 64 || TN == 128, "tile width");
  static_assert(RP == 64 || RP == 128, "padded rank");
  static_assert(!FOLD || (!LOSS && BM == kBmKL), "loss folded into the update kernel: beta 1 only");
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t raw32 = ptx::smem_u32(smem_raw);
  const uint32_t sbase = (raw32 + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (sbase - raw32);
  const uint32_t sF = sbase + L::kF, sG = sbase + L::kG, sV = sbase + L::kV;
  const uint32_t bar0 = sbase + L::kBar;
  auto BAR = [&](int i) { return bar0 + 8u * i; };
  // S/P stage ring: S full (S-MMA -> ratio warps), P full (ratio warps -> O-MMA), P empty (O-MMA -> S-MMA: stage free)
  constexpr int B_FFULL = 0, B_FEMPTY = NF, B_GFULL = 2 * NF, B_GEMPTY = B_GFULL + NG, B_VFULL = B_GEMPTY + NG,
                B_VEMPTY = B_VFULL + NV, B_SFULL = B_VEMPTY + NV, B_PFULL = B_SFULL + NS, B_PEMPTY = B_PFULL + NS,
                B_OFULL = B_PEMPTY + NS, B_OEMPTY = B_OFULL + 1;
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem_al + L::kTmemPtr);
  double* loss_slots = reinterpret_cast<double*>(smem_al + L::kLossSlots);      // [8 ratio warps][2]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == kCtl0 && lane == 0) {
    ptx::prefetch_tmap(&tmF); ptx::prefetch_tmap(&tmG); ptx::prefetch_tmap(&tmV);
    for (int i = 0; i < NF; ++i) { ptx::mbar_init(BAR(B_FFULL + i), 1); ptx::mbar_init(BAR(B_FEMPTY + i), 1); }
    for (int i = 0; i < NG; ++i) { ptx::mbar_init(BAR(B_GFULL + i), 1); ptx::mbar_init(BAR(B_GEMPTY + i), 1); }
    for (int i = 0; i < NV; ++i) { ptx::mbar_init(BAR(B_VFULL + i), 1); ptx::mbar_init(BAR(B_VEMPTY + i), 4 * NRW); }
    for (int i = 0; i < NS; ++i) {
      ptx::mbar_init(BAR(B_SFULL + i), 1); ptx::mbar_init(BAR(B_PFULL + i), 4 * NRW); ptx::mbar_init(BAR(B_PEMPTY + i), 1);
    }
    ptx::mbar_init(BAR(B_OFULL), 1);
    ptx::mbar_init(BAR(B_OEMPTY), 4);
    ptx::fence_barrier_init();
    ptx::fence_proxy_async();
  }
  if (warp == kCtl0 + 1) {
    ptx::tmem_alloc(sbase + L::kTmemPtr, kTmemCols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = *tmem_ptr_smem;

  const int total_items = p.row_blocks * p.nchunks;

  if (warp == kCtl0) {
    // =========================== TMA producer: V tiles (the HBM stream) =================================
    if (lane == 0) {
      uint32_t t = 0;
      for (int item = blockIdx.x; item < total_items; item += gridDim.x) {
        const int rb = item % p.row_blocks, chunk = item / p.row_blocks;
        const int tb = chunk * p.tiles_per_chunk;
        const int te = min(p.tiles, tb + p.tiles_per_chunk);
        for (int j = tb; j < te; ++j, ++t) {
          const uint32_t s = t % NV, ph = (t / NV) & 1;
          ptx::mbar_wait(BAR(B_VEMPTY + s), ph ^ 1);
          ptx::mbar_expect_tx(BAR(B_VFULL + s), L::kVBytes);
          for (int vb = 0; vb < TN / 64; ++vb)
            ptx::tma_load_2d(&tmV, BAR(B_VFULL + s), sV + s * L::kVBytes + vb * (kTileM * 128), j * TN + vb * 64,
                             rb * kTileM);
        }
      }
    }
  } else if (warp == kCtl0 + 2) {
    // =========================== TMA producer: F blocks and G tiles (L2-resident factors) ================
    if (lane == 0) {
      uint32_t it = 0, t = 0;
      for (int item = blockIdx.x; item < total_items; item += gridDim.x, ++it) {
        const int rb = item % p.row_blocks, chunk = item / p.row_blocks;
        const int tb = chunk * p.tiles_per_chunk;
        const int te = min(p.tiles, tb + p.tiles_per_chunk);
        const uint32_t fb = it % NF;
        ptx::mbar_wait(BAR(B_FEMPTY + fb), ((it / NF) & 1) ^ 1);
        ptx::mbar_expect_tx(BAR(B_FFULL + fb), L::kFBytes);
        for (int kb = 0; kb < KW / 64; ++kb)
          ptx::tma_load_2d(&tmF, BAR(B_FFULL + fb), sF + fb * L::kFBytes + kb * (kTileM * 128), kb * 64, rb * kTileM);
        for (int j = tb; j < te; ++j, ++t) {
          const uint32_t s = t % NG, ph = (t / NG) & 1;
          ptx::mbar_wait(BAR(B_GEMPTY + s), ph ^ 1);
          ptx::mbar_expect_tx(BAR(B_GFULL + s), L::kGBytes);
          for (int kb = 0; kb < KW / 64; ++kb)
            ptx::tma_load_2d(&tmG, BAR(B_GFULL + s), sG + s * L::kGBytes + kb * (TN * 128), kb * 64, j * TN);
        }
      }
    }
  } else if (warp == kCtl0 + 1) {
    // =========================== MMA issuer 1: S = F G^T =============================
    // Two issuing warps share the tensor pipe.  An issuing warp is a latency-bound serial instruction stream (barrier
    // polls, descriptor arithmetic in uniform registers, tcgen05.mma issue: measured ~780 cycles per S or O step), so
    // one warp issuing both S and O produced one tile per ~1570 cycles and left the ratio warpgroups waiting for S.
    // This warp runs ahead with the S-MMAs, across work-item boundaries, bounded by the G ring and by the NS
    // accumulator stages (P empty: the O-MMA of the tile NS earlier has consumed the stage); warp 3 issues the O-MMAs as
    // ratio tiles complete.  Each loop is warp-uniform; one elected lane issues tcgen05.mma / commit.
    {
      constexpr uint32_t idescS = ptx::idesc_f16(kTileM, TN, 0, 0);
      constexpr uint32_t descHi = ptx::smem_desc_hi_sw128(1024);
      // S = sum over terms (F part, G part): fast: (0,0); split: (hi,hi), (lo,hi), (hi,lo)
      constexpr int kTerms = SPLIT ? 3 : 1;
      constexpr int termF[3] = {0, 1, 0}, termG[3] = {0, 0, 1};
      uint32_t sg = 0, sg_ph = 0;                 // G stage / phase
      uint32_t ss = 0, ss_ph = 0;                 // S stage / phase of its P-empty barrier
      uint32_t it = 0;
      for (int item = blockIdx.x; item < total_items; item += gridDim.x, ++it) {
        const int tb = (item / p.row_blocks) * p.tiles_per_chunk;
        const int n = min(p.tiles, tb + p.tiles_per_chunk) - tb;
        const uint32_t f_s = it % NF;
        if (lane == 0) ptx::mbar_wait(BAR(B_FFULL + f_s), (it / NF) & 1);       // F block of this item landed
        __syncwarp();      // one poller; the warp is converged again before any elect.sync / tcgen05 issue
        const uint32_t fbase = sF + f_s * L::kFBytes;
        for (int j = 0; j < n; ++j) {
          if (lane == 0) {
            ptx::mbar_wait(BAR(B_GFULL + sg), sg_ph);              // G tile landed
            ptx::mbar_wait(BAR(B_PEMPTY + ss), ss_ph ^ 1);         // the O-MMA of the tile NS earlier consumed its P
          }
          __syncwarp();
          ptx::tc_fence_after();
          const uint32_t gbase = sG + sg * L::kGBytes;
          const uint32_t dS = tmem + kColS + ss * TN;
          if (ptx::elect_one()) {
#pragma unroll
            for (int term = 0; term < kTerms; ++term) {
              // operand halves (hi / lo) are RP/64 sub-blocks of 64 columns each; a k-step is 32 B inside a sub-block
#pragma unroll
              for (int ks = 0; ks < RP / 16; ++ks) {
                const uint32_t alo = ptx::smem_desc_lo(fbase + (termF[term] * (RP / 64) + ks / 4) * (kTileM * 128), 16);
                const uint32_t blo = ptx::smem_desc_lo(gbase + (termG[term] * (RP / 64) + ks / 4) * (TN * 128), 16);
                ptx::mma_ss(dS, ptx::make_desc(alo + 2 * (ks % 4), descHi), ptx::make_desc(blo + 2 * (ks % 4), descHi),
                            idescS, (term | ks) ? 1u : 0u);
              }
            }
            ptx::mma_commit(BAR(B_SFULL + ss));
            if (j == n - 1) ptx::mma_commit(BAR(B_FEMPTY + f_s));  // last S of the item: its F block is free
          }
          __syncwarp();
          if (++sg == NG) { sg = 0; sg_ph ^= 1; }
          if (++ss == NS) { ss = 0; ss_ph ^= 1; }
        }
      }
    }
  } else if (warp == kCtl0 + 3) {
    // =========================== MMA issuer 2: O += P G =============================
    {
      constexpr uint32_t idescO = ptx::idesc_f16(kTileM, KW, 0, 1);
      constexpr uint32_t descHi = ptx::smem_desc_hi_sw128(1024);
      uint32_t og = 0, os = 0, os_ph = 0;         // G stage, S/P stage + phase of its P-full barrier
      uint32_t it = 0;
      for (int item = blockIdx.x; item < total_items; item += gridDim.x, ++it) {
        const int tb = (item / p.row_blocks) * p.tiles_per_chunk;
        const int n = min(p.tiles, tb + p.tiles_per_chunk) - tb;
        for (int j = 0; j < n; ++j) {
          const bool first = j == 0, last = j == n - 1;
          if (lane == 0) {
            ptx::mbar_wait(BAR(B_PFULL + os), os_ph);                              // ratio tile written
            if (first && !LOSS) ptx::mbar_wait(BAR(B_OEMPTY), (it & 1) ^ 1);       // epilogue drained O (none in LOSS mode)
          }
          __syncwarp();
          ptx::tc_fence_after();
          if (LOSS) {
            if (ptx::elect_one()) {                    // nothing to multiply: the ratio warpgroup consumed S, release
              ptx::mbar_arrive(BAR(B_GEMPTY + og));
              ptx::mbar_arrive(BAR(B_PEMPTY + os));
            }
          } else {
            // B = G tile as [K = 16 c-rows][N = KW] MN-major: 8-row groups 1024 B apart, 64-wide column blocks
            // (hi | lo, RP/64 blocks each) one sub-block (TN x 128 B) apart
            const uint32_t blo = ptx::smem_desc_lo(sG + og * L::kGBytes, TN * 128);
            const uint32_t aP = tmem + kColS + os * TN;
            if (ptx::elect_one()) {
#pragma unroll
              for (int ks = 0; ks < TN / 16; ++ks) {
                // P k-step ks was written by ratio warpgroup ks / kKsPerWg, at the start of that warpgroup's S columns
                constexpr int kKsPerWg = TN / 16 / NRW;
                ptx::mma_ts(tmem + kColO, aP + (ks / kKsPerWg) * (TN / NRW) + (ks % kKsPerWg) * 8,
                            ptx::make_desc(blo + ks * 128, descHi), idescO, (first && ks == 0) ? 0u : 1u);
                if (TWO)
                  ptx::mma_ts(tmem + kColO2, tmem + kColPp + os * 64 + ks * 8, ptx::make_desc(blo + ks * 128, descHi),
                              idescO, (first && ks == 0) ? 0u : 1u);
              }
              ptx::mma_commit(BAR(B_GEMPTY + og));     // G tile free (its S-MMA finished before the ratio tile existed)
              ptx::mma_commit(BAR(B_PEMPTY + os));     // S/P stage free
              if (last) ptx::mma_commit(BAR(B_OFULL));
            }
          }
          __syncwarp();
          if (++og == NG) og = 0;
          if (++os == NS) { os = 0; os_ph ^= 1; }
        }
      }
    }
  } else if (warp < kEpiWarp0) {
    // =========================== ratio warpgroups =======================
    // Every tile is split by COLUMNS between the NRW ratio warpgroups (each covers all 128 TMEM lanes): the time a tile
    // spends in the ratio stage is what holds its S/P accumulator stage, and with NS = 3 stages that hold time -- not
    // MUFU, shared-memory or HBM throughput -- set the tile period (knock-out timing, DESIGN.md 4.1).  Splitting a
    // tile halves the hold; alternating whole tiles between the warpgroups did not.
    const int g = warp >> 2;                   // this warpgroup handles columns [g TN / NRW, (g + 1) TN / NRW) of every tile
    const int q = warp & 3;                    // TMEM lane quarter this warp may touch
    const int row = q * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const int ev = p.exps[0], ea = p.exps[p.ef], eb = p.exps[p.eg], ep = p.exps[3];
    // update: x' = (S + eps) * 2^(v-p), so P~ = V~ / x' = P * 2^p (P ~ 1 maps to ~1: fp16-safe for any input scale)
    // loss  : x  = S + eps in true scale
    const float c1 = (LOSS || TWO) ? exp2f((float)(-ea - eb)) : exp2f((float)(ev - ea - eb - ep));
    const float c2 = (LOSS || TWO) ? kEps : kEps * exp2f((float)(ev - ep));
    // two-output kernels: Pn~ = V~ x^(beta-2) kn, Pp~ = x^(beta-1) kd with x = S + eps in true scale
    const float kn = TWO ? exp2f((float)(p.exps[4] - ev)) : 0.f;
    const float kd = TWO ? exp2f((float)p.exps[5]) : 0.f;
    // The tile fed to MMA-2 is the CENTRED ratio (P - kappa) 2^p with kappa = sum(V) / sum(W H^T) (-> 1 as the fit
    // converges); kappa * colsum(G) is added back in fp32 by the ratio stage.  Tensor-core accumulation truncates
    // (measured: -4.7e-5 relative on this all-positive sum, profiles/README.md), a one-signed bias that the
    // scale-free direction (W a, H / a) of KL-NMF integrates over iterations; the centred sum is signed and
    // small, and its fp16 rounding error is relative to |P - kappa| instead of |P|.
    const float negpc = (LOSS || TWO || EU) ? 0.f : -(*p.kappa) * exp2f((float)ep);
    // beta 2: P~ = (V - WH) 2^pe = v~ cv - s~ cs   (pe = exps[4], from mean(V)); loss: true scale (pe = 0)
    const float eu_cv = EU ? exp2f((float)((LOSS ? 0 : p.exps[4]) - ev)) : 0.f;
    // update: the tile is V - kappa WH with kappa = sum(V) / sum(WH) (the scale-matched residual; kappa -> 1 as the fit
    // converges), so that far from convergence (WH >> V) the numerator is not a small difference of large sums
    const float eu_cs = EU ? exp2f((float)((LOSS ? 0 : p.exps[4]) - ea - eb)) * (LOSS ? 1.f : *p.kappa) : 0.f;
    double accA = 0.0, accB = 0.0;
    uint32_t t = 0;
    const float vinv = exp2f(-(float)ev);
    if constexpr (!LOSS && !TWO) {
      // ---- update tiles of beta 1 / beta 2: ONE flat software pipeline over every (tile, 16-column chunk) of this CTA.
      // The stage is bound by the FMA pipe of the four SM sub-partitions, not by latency (measured, tools/ubench/pipes.cu on
      // the B200: FFMA 1.6, FFMA2 2.3, FMUL2 3.7, HFMA2 2.0, IMAD / LOP3 / PRMT 2.1, MUFU 8.0 cycles per warp instruction and
      // sub-partition; four ratio warpgroups instead of two changed nothing).  Hence:
      // * everything runs as packed fp32 pairs through FFMA2 (a product is an FFMA2 with a zero addend: FMUL2 is slower);
      // * three quarters of the reciprocals are batched four elements to two MUFU ops (1/a = b rcp(a b): +3 FFMA2 per four
      //   elements, -2 MUFU), which balances the XU pipe (640 cycles per tile) against the FMA pipe (~690);
      // * addresses are formed once per tile (swizzled shared-memory offsets by one XOR with a constant per load), ring
      //   positions are counted, not divided;
      // * the TMEM load of S and the shared-memory load of V for chunk c + 1 are in flight while chunk c is computed, across
      //   tile boundaries (the next tile's first chunk is requested before this tile's last chunk is computed).
      // A "chunk" is CW columns of the tile: the unit of the load / compute software pipeline (the loads of chunk c + 1 are in
      // flight while chunk c is computed).  32-column chunks (twice the lookahead, 126 registers) measured slower than 16
      // (116 / 122 us vs 111 / 118 us per launch at cfg2): the stage is not waiting for its loads.
      constexpr int CW = 16;                                    // tmem_ld16 / tmem_st8 below
      constexpr int kChunks = TN / CW;
      constexpr int kCpw = kChunks / NRW;                       // chunks per warpgroup and tile
      static_assert(kCpw % 2 == 0 && kChunks % NRW == 0, "chunks per ratio warpgroup");
      const int c_lo = g * kCpw;
      uint32_t my_tiles = 0;
      for (int item = blockIdx.x; item < total_items; item += gridDim.x) {
        const int tb = (item / p.row_blocks) * p.tiles_per_chunk;
        my_tiles += min(p.tiles, tb + p.tiles_per_chunk) - tb;
      }
      const uint64_t C1 = ptx::pk2(c1, c1), C2 = ptx::pk2(c2, c2), NEGPC = ptx::pk2(negpc, negpc), Z2 = ptx::pk2(0.f, 0.f);
      const uint64_t EUCV = ptx::pk2(eu_cv, eu_cv), EUNCS = ptx::pk2(-eu_cs, -eu_cs);
      // FOLD: x = WH + eps in true scale (the LOSS kernel's c1 / c2), sum v~ lg2 x and sum S~ of this thread and tile
      const float c1l = exp2f((float)(-ea - eb));
      const uint64_t C1L = ptx::pk2(c1l, c1l), C2L = ptx::pk2(kEps, kEps), ONE2 = ptx::pk2(1.f, 1.f);
      float fold_a = 0.f;
      uint64_t FOLD_B = Z2;
      // this thread's row inside a 128-byte-swizzled V sub-tile: byte (row, 16-byte chunk k) sits at row*128 + ((k ^ row%8) << 4)
      const uint32_t vrow = (uint32_t)row * 128u + ((uint32_t)(row & 7) << 4);
      const uint32_t tS0 = tmem + lane_addr + kColS;            // TMEM address of this warp's lanes, stage 0, column 0
      constexpr int NV4 = CW / 8;                               // 16-byte shared-memory loads per chunk
      uint32_t sA[CW], sB[CW];
      uint4 vA[NV4], vB[NV4];
      auto load_chunk = [&](uint32_t tS, uint32_t vT, int c, uint32_t (&sr)[CW], uint4 (&vv)[NV4]) {
        ptx::tmem_ld16(tS + c * CW, sr);
#pragma unroll
        for (int k = 0; k < NV4; ++k) {
          const int col16 = c * NV4 + k;                                           // 16-byte column group of the tile (8 fp16)
          const uint32_t kx = (uint32_t)(col16 & 7) << 4;                          // compile-time per unrolled load
          asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                       : "=r"(vv[k].x), "=r"(vv[k].y), "=r"(vv[k].z), "=r"(vv[k].w)
                       : "r"((vT ^ kx) + (uint32_t)((col16 >> 3) * (kTileM * 128))));
        }
      };
      auto compute_chunk = [&](uint32_t tS, int c, const uint32_t (&sr)[CW], const uint4 (&vv)[NV4]) {
        const uint32_t* vw = reinterpret_cast<const uint32_t*>(vv);
        uint32_t preg[CW / 2];
#pragma unroll
        for (int qd = 0; qd < CW / 4; ++qd) {                    // four consecutive columns: pairs a = (0, 1), b = (2, 3)
          const float2 va = __half22float2(*reinterpret_cast<const __half2*>(&vw[2 * qd]));
          const float2 vb = __half22float2(*reinterpret_cast<const __half2*>(&vw[2 * qd + 1]));
          const uint64_t Va = ptx::pk2(va.x, va.y), Vb = ptx::pk2(vb.x, vb.y);
          const uint64_t Sa = ptx::pk2(__uint_as_float(sr[4 * qd]), __uint_as_float(sr[4 * qd + 1]));
          const uint64_t Sb = ptx::pk2(__uint_as_float(sr[4 * qd + 2]), __uint_as_float(sr[4 * qd + 3]));
          uint64_t Pa, Pb;
          if (EU) {
            Pa = ptx::fma2(Sa, EUNCS, ptx::fma2(Va, EUCV, Z2));                       // nmf.py:62-63: V - kappa WH
            Pb = ptx::fma2(Sb, EUNCS, ptx::fma2(Vb, EUCV, Z2));
          } else {
            const uint64_t Xa = ptx::fma2(Sa, C1, C2), Xb = ptx::fma2(Sb, C1, C2);   // (WH + eps) in the scale of V~ / P~
            if constexpr (FOLD) {                                                    // metrics.py:22 on the same S tile
              float l0, l1, l2, l3;
              ptx::upk2(ptx::fma2(Sa, C1L, C2L), l0, l1);
              ptx::upk2(ptx::fma2(Sb, C1L, C2L), l2, l3);
              fold_a = fmaf(va.x, __log2f(l0), fold_a);
              fold_a = fmaf(va.y, __log2f(l1), fold_a);
              fold_a = fmaf(vb.x, __log2f(l2), fold_a);
              fold_a = fmaf(vb.y, __log2f(l3), fold_a);
              FOLD_B = ptx::fma2(Sa, ONE2, FOLD_B);
              FOLD_B = ptx::fma2(Sb, ONE2, FOLD_B);
            }
            uint64_t Ra, Rb;                                                         // 1 / x of pair a, pair b
            if ((qd & 3) != 0) {
              // batched: 1 / x0 = x2 r0, 1 / x1 = x3 r1, 1 / x2 = x0 r0, 1 / x3 = x1 r1 with r = rcp(x_a x_b)
              float m0, m1;
              ptx::upk2(ptx::fma2(Xa, Xb, Z2), m0, m1);
              const uint64_t Rr = ptx::pk2(ptx::rcp_approx(m0), ptx::rcp_approx(m1));
              Ra = ptx::fma2(Rr, Xb, Z2);
              Rb = ptx::fma2(Rr, Xa, Z2);
            } else {
              float x0, x1, x2, x3;
              ptx::upk2(Xa, x0, x1);
              ptx::upk2(Xb, x2, x3);
              Ra = ptx::pk2(ptx::rcp_approx(x0), ptx::rcp_approx(x1));
              Rb = ptx::pk2(ptx::rcp_approx(x2), ptx::rcp_approx(x3));
            }
            Pa = ptx::fma2(Va, Ra, NEGPC);                                           // nmf.py:65, centred
            Pb = ptx::fma2(Vb, Rb, NEGPC);
          }
          float a0, a1, b0, b1;
          ptx::upk2(Pa, a0, a1);
          ptx::upk2(Pb, b0, b1);
          preg[2 * qd] = ptx::pack_f16x2_sat(a0, a1);
          preg[2 * qd + 1] = ptx::pack_f16x2_sat(b0, b1);
        }
        // P of warpgroup g goes over the S columns that warpgroup owns (and has already read): [g TN / NRW, ...)
        ptx::tmem_st8(tS + g * (TN / NRW) + (c - c_lo) * (CW / 2), preg);
      };
      uint32_t st = 0, sv = 0, phS = 0, phV = 0;        // S stage and V slot of the tile being computed, phases of their full barriers
      uint32_t tS = tS0, vT = sV + vrow;
      if (my_tiles > 0) {
        ptx::mbar_wait(BAR(B_VFULL), 0);                            // V tile landed (TMA -> this thread)
        ptx::mbar_wait(BAR(B_SFULL), 0);                            // S tile complete
        ptx::tc_fence_after();
        load_chunk(tS, vT, c_lo, sA, vA);
      }
      for (uint32_t tt = 0; tt < my_tiles; ++tt) {
        const bool more = tt + 1 < my_tiles;
        // ring positions of the next tile
        uint32_t st1 = st + 1, phS1 = phS, sv1 = sv + 1, phV1 = phV;
        if (st1 == NS) { st1 = 0; phS1 ^= 1; }
        if (sv1 == NV) { sv1 = 0; phV1 ^= 1; }
        const uint32_t tS1 = tS0 + st1 * TN, vT1 = sV + sv1 * L::kVBytes + vrow;
#pragma unroll
        for (int cc = 0; cc < kCpw; cc += 2) {
          const int c = c_lo + cc;
          const bool lastpair = cc + 2 >= kCpw;
          // The next tile's full barriers are TESTED a chunk of work before they are needed: a try_wait returns its answer
          // after ~100 cycles even when the phase completed long ago (ncu source page: 15 % of the ratio warps' time sat on
          // the two polls of every tile), and both ratio warps of a sub-partition reach them together.
          bool okV = false, okS = false;
          if (lastpair && more) {
            okV = ptx::mbar_test_wait(BAR(B_VFULL + sv1), phV1);
            okS = ptx::mbar_test_wait(BAR(B_SFULL + st1), phS1);
          }
          ptx::tc_wait_ld();
          load_chunk(tS, vT, c + 1, sB, vB);
          compute_chunk(tS, c, sA, vA);
          ptx::tc_wait_ld();
          if (!lastpair) {
            load_chunk(tS, vT, c + 2, sA, vA);
          } else if (more) {
            if (!okV) ptx::mbar_wait(BAR(B_VFULL + sv1), phV1);
            if (!okS) ptx::mbar_wait(BAR(B_SFULL + st1), phS1);
            ptx::tc_fence_after();
            load_chunk(tS1, vT1, c_lo, sA, vA);
          }
          compute_chunk(tS, c + 1, sB, vB);
        }
        // hand the tile on: P complete (this also frees the S stage once the O-MMA has run) + the V slot
        ptx::tc_wait_st();
        ptx::tc_fence_before();
        __syncwarp();                  // every lane's P stores are complete and fenced, its V reads have returned
        if (lane == 0) {               // ONE arrival per warp (barrier counts = warps): 32x fewer mbarrier operations
          ptx::mbar_arrive(BAR(B_PFULL + st));
          ptx::mbar_arrive(BAR(B_VEMPTY + sv));
        }
        st = st1; phS = phS1; sv = sv1; phV = phV1; tS = tS1; vT = vT1;
        if constexpr (FOLD) {                    // per-tile fp32 sums (TN / NRW elements per thread) into the double totals
          float b0, b1;
          ptx::upk2(FOLD_B, b0, b1);
          accA += (double)fold_a;
          accB += (double)(b0 + b1);
          fold_a = 0.f;
          FOLD_B = Z2;
        }
      }
    } else {
    for (int item = blockIdx.x; item < total_items; item += gridDim.x) {
      const int chunk = item / p.row_blocks;
      const int tb = chunk * p.tiles_per_chunk;
      const int te = min(p.tiles, tb + p.tiles_per_chunk);
      const int n = te - tb;
      const bool row_ok = (item % p.row_blocks) * kTileM + row < p.Mr;
      for (int j = 0; j < n; ++j) {
        const uint32_t tt = t + j;
        const uint32_t s = tt % NV, st = tt % NS;
        ptx::mbar_wait(BAR(B_VFULL + s), (tt / NV) & 1);              // V tile landed (TMA -> this thread)
        ptx::mbar_wait(BAR(B_SFULL + st), (tt / NS) & 1);       // S tile complete
        ptx::tc_fence_after();
        const uint32_t vrow = sV + s * L::kVBytes + row * 128;
        {
#pragma unroll
        for (int c4r = 0; c4r < TN / 32 / NRW; ++c4r) {
          const int c4 = g * (TN / 32 / NRW) + c4r;
          uint32_t sreg[32];
          ptx::tmem_ld32(tmem + lane_addr + kColS + st * TN + c4 * 32, sreg);
          uint4 vv[4];
          const uint32_t vsub = vrow + (c4 >> 1) * (kTileM * 128);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint32_t chunk16 = (uint32_t)((c4 & 1) * 4 + k) ^ (uint32_t)(row & 7);
            asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(vv[k].x), "=r"(vv[k].y), "=r"(vv[k].z), "=r"(vv[k].w)
                         : "r"(vsub + (chunk16 << 4)));
          }
          ptx::tc_wait_ld();
          const uint32_t* vw = reinterpret_cast<const uint32_t*>(vv);
          if (LOSS && EU) {
            float la = 0.f;                        // metrics.py:39: 0.5 sum (WH - V)^2 (zero-filled edges contribute 0)
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float2 vf = __half22float2(*reinterpret_cast<const __half2*>(&vw[i]));
              const float d0 = fmaf(vf.x, eu_cv, -__uint_as_float(sreg[2 * i]) * eu_cs);
              const float d1 = fmaf(vf.y, eu_cv, -__uint_as_float(sreg[2 * i + 1]) * eu_cs);
              la = fmaf(d0, d0, la);
              la = fmaf(d1, d1, la);
            }
            accA += (double)la;
          } else if (LOSS && BM == kBmKL) {
            float la = 0.f, lb = 0.f;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float2 vf = __half22float2(*reinterpret_cast<const __half2*>(&vw[i]));
              const float s0 = __uint_as_float(sreg[2 * i]), s1 = __uint_as_float(sreg[2 * i + 1]);
              la = fmaf(vf.x, __log2f(fmaf(s0, c1, c2)), la);
              la = fmaf(vf.y, __log2f(fmaf(s1, c1, c2)), la);
              lb += s0 + s1;
            }
            accA += (double)la;
            accB += (double)lb;
          } else if (LOSS) {
            // metrics.py:56-57 (beta 0) and :84-96 (generic): A = sum t x^(beta-1), B = sum x^beta (beta 0: sum ln x / ln 2).
            // Out-of-range rows / columns are zero-filled operands (x = eps there) and must be masked out.
            float la = 0.f, lb = 0.f;
            const int col0 = (tb + j) * TN + c4 * 32;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float2 vf = __half22float2(*reinterpret_cast<const __half2*>(&vw[i]));
#pragma unroll
              for (int e = 0; e < 2; ++e) {
                const bool ok = row_ok && col0 + 2 * i + e < p.Nc;
                const float x = fmaf(__uint_as_float(sreg[2 * i + e]), c1, c2);
                const float v = (e ? vf.y : vf.x) * vinv;
                const float lx = __log2f(x);
                float ta, tb2;
                if (BM == kBmIS) {
                  ta = (v + kEps) * ptx::rcp_approx(x);
                  tb2 = lx;
                } else {
                  const float tv = p.bm1 < -1.f ? v + kEps : v;          // beta < 0: target + eps (metrics.py:87-88)
                  ta = tv * exp2f(p.bm1 * lx);
                  tb2 = exp2f((p.bm1 + 1.f) * lx);
                }
                la += ok ? ta : 0.f;
                lb += ok ? tb2 : 0.f;
              }
            }
            accA += (double)la;
            accB += (double)lb;
          } else if (TWO) {
            uint32_t pn[16], pp[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float2 vf = __half22float2(*reinterpret_cast<const __half2*>(&vw[i]));
              float fn[2], fp[2];
#pragma unroll
              for (int e = 0; e < 2; ++e) {
                const float x = fmaf(__uint_as_float(sreg[2 * i + e]), c1, c2);        // WH + eps, nmf.py:68,72
                if (BM == kBmIS) {                 // nmf.py:68-70
                  const float r = ptx::rcp_approx(x);
                  fp[e] = r; fn[e] = r * r;
                } else if (BM == kBm05) {          // x^-0.5, x^-1.5
                  const float rs = rsqrtf(x);
                  fp[e] = rs; fn[e] = rs * rs * rs;
                } else if (BM == kBm15) {          // x^0.5, x^-0.5
                  const float rs = rsqrtf(x);
                  fp[e] = x * rs; fn[e] = rs;
                } else {                           // nmf.py:72-74
                  const float l = __log2f(x);
                  fp[e] = exp2f(p.bm1 * l); fn[e] = exp2f(p.bm2 * l);
                }
              }
              pn[i] = ptx::pack_f16x2_sat(vf.x * fn[0] * kn, vf.y * fn[1] * kn);
              pp[i] = ptx::pack_f16x2_sat(fp[0] * kd, fp[1] * kd);
            }
            ptx::tmem_st16(tmem + lane_addr + kColS + st * TN + g * (TN / NRW) + c4r * 16, pn);   // own S columns, see above
            ptx::tmem_st16(tmem + lane_addr + kColPp + st * 64 + c4 * 16, pp);
          }
        }
        }
        if (!LOSS) ptx::tc_wait_st();
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          ptx::mbar_arrive(BAR(B_PFULL + st));
          ptx::mbar_arrive(BAR(B_VEMPTY + s));
        }
      }
      t += n;
    }
    }   // LOSS and two-output kernels
    if (LOSS || FOLD) {
      for (int o = 16; o > 0; o >>= 1) {
        accA += __shfl_xor_sync(0xffffffffu, accA, o);
        accB += __shfl_xor_sync(0xffffffffu, accB, o);
      }
      if (lane == 0) { loss_slots[2 * warp] = accA; loss_slots[2 * warp + 1] = accB; }
    }
  } else if (warp >= kEpiWarp0 && warp < kCtl0 && !LOSS) {
    // =========================== epilogue warpgroup =====================
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const float oscale = exp2f(-(float)(p.exps[p.eg] + p.exps[(TWO || EU) ? 4 : 3]));      // O = sum (P 2^p) (G 2^eg)
    const float oscale2 = TWO ? exp2f(-(float)(p.exps[p.eg] + p.exps[5])) : 0.f;
    uint32_t it = 0;
    for (int item = blockIdx.x; item < total_items; item += gridDim.x, ++it) {
      const int rb = item % p.row_blocks, chunk = item / p.row_blocks;
      if (lane == 0) ptx::mbar_wait(BAR(B_OFULL), it & 1);      // one polling lane per warp
      __syncwarp();
      ptx::tc_fence_after();
      const int64_t grow = (int64_t)rb * kTileM + row;
      float* dst = p.part + (int64_t)chunk * p.chunk_stride + grow * p.ldp;
      if (TWO) {
        // numerator then denominator accumulator (64 columns each); O is handed back after the last TMEM load
        float* dst2 = p.part2 + (int64_t)chunk * p.chunk_stride + grow * p.ldp;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          float o[64];
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            uint32_t raw[32];
            ptx::tmem_ld32(tmem + lane_addr + (half ? kColO2 : kColO) + c * 32, raw);
            ptx::tc_wait_ld();
#pragma unroll
            for (int i = 0; i < 32; ++i) o[c * 32 + i] = __uint_as_float(raw[i]) * (half ? oscale2 : oscale);
          }
          if (half == 1) { ptx::tc_fence_before(); __syncwarp(); if (lane == 0) ptx::mbar_arrive(BAR(B_OEMPTY)); }
          if (grow < p.Mr) {
            float* d = half ? dst2 : dst;
#pragma unroll
            for (int i = 0; i < 64; i += 4) *reinterpret_cast<float4*>(d + i) = make_float4(o[i], o[i + 1], o[i + 2], o[i + 3]);
          }
        }
        continue;
      }
      if (RP == 64) {
        // whole O row (64 values) into registers, hand the accumulator back to the MMA warp, then store
        float o[64];
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          uint32_t hi[32];
          ptx::tmem_ld32(tmem + lane_addr + kColO + c * 32, hi);
          if (SPLIT) {
            uint32_t lo[32];
            ptx::tmem_ld32(tmem + lane_addr + kColO + RP + c * 32, lo);
            ptx::tc_wait_ld();
#pragma unroll
            for (int i = 0; i < 32; ++i) o[c * 32 + i] = (__uint_as_float(hi[i]) + __uint_as_float(lo[i])) * oscale;
          } else {
            ptx::tc_wait_ld();
#pragma unroll
            for (int i = 0; i < 32; ++i) o[c * 32 + i] = __uint_as_float(hi[i]) * oscale;
          }
        }
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(BAR(B_OEMPTY));
        // Each lane owns a row, so one store instruction touches 32 cache lines = 32 passes through the load/store unit
        // that the ratio warps' shared-memory loads (and every other memory instruction of the SM) queue behind: issued
        // back to back, the 64 stores of an item stopped the whole SM for ~2300 cycles at every item boundary (per-tile
        // trace: 9 % of the launch).  Nothing waits for these stores (the next epilogue is 16 tiles away): pace them.
        if (grow < p.Mr) {
#pragma unroll
          for (int i = 0; i < 64; i += 8) {          // 256-bit stores: half the instructions, half the passes
            asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                         ::"l"(dst + i), "f"(o[i]), "f"(o[i + 1]), "f"(o[i + 2]), "f"(o[i + 3]), "f"(o[i + 4]), "f"(o[i + 5]),
                           "f"(o[i + 6]), "f"(o[i + 7]) : "memory");
            __nanosleep(kEpiPaceNs);
          }
        }
        continue;
      }
#pragma unroll
      for (int c = 0; c < RP / 32; ++c) {
        uint32_t hi[32];
        ptx::tmem_ld32(tmem + lane_addr + kColO + c * 32, hi);
        float o[32];
        if (SPLIT) {
          uint32_t lo[32];
          ptx::tmem_ld32(tmem + lane_addr + kColO + RP + c * 32, lo);
          ptx::tc_wait_ld();
#pragma unroll
          for (int i = 0; i < 32; ++i) o[i] = (__uint_as_float(hi[i]) + __uint_as_float(lo[i])) * oscale;
        } else {
          ptx::tc_wait_ld();
#pragma unroll
          for (int i = 0; i < 32; ++i) o[i] = __uint_as_float(hi[i]) * oscale;
        }
        if (grow < p.Mr) {
#pragma unroll
          for (int i = 0; i < 32; i += 4)
            *reinterpret_cast<float4*>(dst + c * 32 + i) = make_float4(o[i], o[i + 1], o[i + 2], o[i + 3]);
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(BAR(B_OEMPTY));
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == kCtl0 + 1) ptx::tmem_dealloc(tmem, kTmemCols);
  if ((LOSS || FOLD) && threadIdx.x == (kCtl0 + 3) * 32) {          // fixed-order sum of the 8 ratio warps
    double a = 0.0, b = 0.0;
    for (int w = 0; w < 4 * NRW; ++w) { a += loss_slots[2 * w]; b += loss_slots[2 * w + 1]; }
    p.loss_part[2 * blockIdx.x] = a;
    p.loss_part[2 * blockIdx.x + 1] = b;
  }
}

// ---- operand preparation --------------------------------------------------------------------------

__device__ __forceinline__ int pow2_exp_for(float mx) {
  // exponent a with mx * 2^a in [2^13, 2^14); 0 for an all-zero / non-finite matrix
  if (!(mx > 0.f) || !isfinite(mx)) return 0;
  int e;
  frexpf(mx, &e);               // mx = m * 2^e, m in [0.5, 1)
  return 14 - e;
}

// What the last stage of a factor refresh publishes (one thread): the operand exponent of this factor, kappa =
// sum(V) / sum(W H^T) = sum(V) / <colsum W, colsum H> (the typical P = V / (WH)), the ratio-tile exponent exps[3] with
// kappa 2^p in [2^-4, 2^-3) (P - kappa is fp16-exact down to 2^-20 kappa, and a ratio has to exceed 5e5 kappa before the
// saturating pack clips it), and the exponents of the beta != 1 tiles.
__device__ __forceinline__ void publish_scales(int a, int which, int* __restrict__ exps, unsigned int* __restrict__ absmax_next,
                                               float dot, const double* __restrict__ vconst, float* __restrict__ kappa,
                                               int center, float bm1, float bm2, double cells) {
  exps[1 + which] = a;
  *absmax_next = 0u;
  const float ptyp = (float)(vconst[0] / (double)dot);
  int e = 0;
  const bool ok = ptyp > 0.f && isfinite(ptyp);
  if (ok) { frexpf(ptyp, &e); e = -3 - e; }     // ptyp * 2^e in [2^-4, 2^-3)
  exps[3] = e;
  *kappa = (ok && center) ? ptyp : 0.f;
  // beta != 1: typical x = mean(WH), typical Pn = mean(V) x^(beta-2), Pp = x^(beta-1) -> both tiles near 2^0
  const float xbar = (float)((double)dot / cells), vbar = (float)(vconst[0] / cells);
  int en = 0, ed = 0;
  if (xbar > 0.f && isfinite(xbar)) {
    const float lx = log2f(xbar);
    const float ln = (vbar > 0.f ? log2f(vbar) : 0.f) + bm2 * lx, ld = bm1 * lx;
    if (isfinite(ln)) en = -(int)rintf(ln);
    if (isfinite(ld)) ed = -(int)rintf(ld);
  }
  exps[4] = en;
  exps[5] = ed;
}

__global__ void set_vexp_kernel(const float* __restrict__ minmax, int* __restrict__ exps) {
  if (threadIdx.x == 0 && blockIdx.x == 0) exps[0] = pow2_exp_for(minmax[1]);
}

__device__ __forceinline__ double block_sum256(double v, double* sh) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x < 32) {
    t = threadIdx.x < 8 ? sh[threadIdx.x] : 0.0;
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  }
  __syncthreads();
  return t;     // valid in warp 0
}

// V (N x C fp32, ld) -> V16 (N x ldc) and Vt16 (C x ldn), both scaled by 2^exps[0]; 64x64 tiles.
// Also per-block partial sums of V and V*log(V+eps) (the V-only terms of metrics.kl_div, metrics.py:22).
__global__ void __launch_bounds__(256)
v_to_f16_kernel(const float* __restrict__ V, int64_t ldv, int N, int C, __half* __restrict__ V16, int64_t ldc,
                __half* __restrict__ Vt16, int64_t ldn, const int* __restrict__ exps, double* __restrict__ vpart,
                unsigned long long* __restrict__ lossy) {
  __shared__ float tile[64][65];
  __shared__ double red[8];
  const float sc = exp2f((float)exps[0]);
  const int n0 = blockIdx.y * 64, c0 = blockIdx.x * 64;
  double sv = 0.0, svl = 0.0;
  unsigned int nlossy = 0;      // positive entries below the fp16 normal range of the scaled copy (subnormal or flushed)
  for (int idx = threadIdx.x; idx < 64 * 64; idx += 256) {
    int r = idx >> 6, c = idx & 63;
    const bool in = n0 + r < N && c0 + c < C;
    const float raw = in ? V[(int64_t)(n0 + r) * ldv + c0 + c] : 0.f;
    const float v = raw * sc;
    tile[r][c] = v;
    if (in) {
      V16[(int64_t)(n0 + r) * ldc + c0 + c] = __float2half_rn(v);
      nlossy += (raw > 0.f && v < 6.103515625e-05f) ? 1u : 0u;
      sv += (double)raw;
      svl += (double)(raw * logf(raw + kEps));
    }
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < 64 * 64; idx += 256) {
    int c = idx >> 6, r = idx & 63;
    if (n0 + r < N && c0 + c < C) Vt16[(int64_t)(c0 + c) * ldn + n0 + r] = __float2half_rn(tile[r][c]);
  }
  const int64_t blk = (int64_t)blockIdx.y * gridDim.x + blockIdx.x;
  double a = block_sum256(sv, red);
  double b = block_sum256(svl, red);
  if (threadIdx.x == 0) { vpart[2 * blk] = a; vpart[2 * blk + 1] = b; }
  nlossy = __reduce_add_sync(0xffffffffu, nlossy);
  if ((threadIdx.x & 31) == 0 && nlossy) atomicAdd(lossy, (unsigned long long)nlossy);
}

// vconst[0] = sum V, vconst[1] = sum V log(V + eps): fixed-order two-level reduction (single block)
__global__ void __launch_bounds__(256)
reduce_vconst_kernel(const double* __restrict__ vpart, int64_t nblk, double* __restrict__ vconst) {
  __shared__ double red[8];
  double a = 0.0, b = 0.0;
  for (int64_t i = threadIdx.x; i < nblk; i += 256) { a += vpart[2 * i]; b += vpart[2 * i + 1]; }
  double ta = block_sum256(a, red);
  double tb = block_sum256(b, red);
  if (threadIdx.x == 0) { vconst[0] = ta; vconst[1] = tb; }
}

// ---- fused ratio stage for the tensor-core path (nmf.py:78-92, KL: precomputed denominator) -------------
// grid = ceil(rows / rpb); 256 threads = 4 row groups x 64 rank lanes.  Besides the in-place update it emits
// what the next kernels need: per-block column sums (-> KL denominator of the other factor) and the max
// (-> power-of-two scale of the fp16 operand copy).
constexpr int kMaxPeers = 8;      // ranks of one NVLink domain that may share a W update

struct TcApplyArgs {
  float* param; int64_t rows; int R; int rpb;
  const float* num; int nchunks; int64_t chunk_stride; int Rp;     // partial row pitch = padded rank
  const float* den;          // beta != 1: partial denominators (same layout); nullptr for beta == 1
  const float* kl_den; float gamma, l1, l2;
  float* cs_part;            // [gridDim.x][128]
  const float* kappa;        // the kernel accumulated sum (P - kappa) G: add kappa * colsum(G) back
  unsigned int* absmax;      // slot to atomicMax into (pre-zeroed)
  int apply;                 // 0: only emit column sums / max of the current values (dirty-factor resync)
  // Row-sharded W update over peer memory (NVLink): the numerator is the sum, in rank order, of every rank's packed buffer
  // [rows x R | R or rows x R], read with P2P loads once every rank has published this iteration's counter in `flags`.
  const float* peers[kMaxPeers]; int npeers; const unsigned int* flags; unsigned int flag_target; unsigned int* peer_err;
};

__global__ void __launch_bounds__(256)
tc_apply_kernel(TcApplyArgs a) {
  __shared__ float sh[2][128];
  const int r = threadIdx.x & 127, rg = threadIdx.x >> 7;
  const int64_t row0 = (int64_t)blockIdx.x * a.rpb;
  const int64_t row1 = min(a.rows, row0 + a.rpb);
  float cs = 0.f, mx = 0.f;
  if (r < a.R) {
    const float klden = (a.apply && !a.den) ? a.kl_den[r] : 1.f;
    const float kap = (a.apply && !a.den) ? *a.kappa : 0.f;
    for (int64_t row = row0 + rg; row < row1; row += 2) {
      const int64_t idx = row * a.R + r;
      float v = a.param[idx];
      if (a.apply) {
        float num = 0.f;
        for (int ch = 0; ch < a.nchunks; ++ch) num += a.num[ch * a.chunk_stride + row * a.Rp + r];
        float pos;
        if (a.den) {
          float den = 0.f;
          for (int ch = 0; ch < a.nchunks; ++ch) den += a.den[ch * a.chunk_stride + row * a.Rp + r];
          pos = fmaxf(den, 0.f) + kEps;                         // nmf.py:83
        } else {
          num = fmaf(kap, klden, num);                          // the kernel accumulated sum (P - kappa) G
          pos = klden;                                          // nmf.py:368-369 / :381-382
        }
        v = mu_step(v, num, pos, a.l1, a.l2, a.gamma);
        a.param[idx] = v;
      }
      cs += v;
      mx = fmaxf(mx, v);
    }
  }
  sh[rg][r] = cs;
  __syncthreads();
  if (threadIdx.x < 128) a.cs_part[(int64_t)blockIdx.x * 128 + r] = sh[0][r] + sh[1][r];
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0 && mx > 0.f) atomicMax(a.absmax, __float_as_uint(mx));
}

// beta 2 denominators.  gram_part_kernel: per-slab partial G^T G (R x R, fp32); gram_sum_kernel folds the slabs in
// fixed order.  tc_apply_eu_kernel: den_raw = F (G^T G) row by row (the reference's relu(S^T G), nmf.py:63,82, since
// S = F G^T), num = O + den_raw with O = (V - S)-contraction from the tensor cores, then nmf.py:78-92.
//
// Both are small dense products (cfg5: 2.7e8 FMA each) and both were one-output-per-thread loops with two shared-memory
// loads per FMA: ~100 us each at 65536 x 64, more than the tensor-core contraction they accompany (beta 2 ran at 570 us per
// iteration with 211 us of contractions).  They are register-tiled now: a thread owns a TR x TR (Gram) or 4 x TR (ratio
// stage) block of outputs, TR = Rp / 16, so that one 16-byte and a few broadcast loads feed 16 to 64 FMAs.
template <int TR>
__global__ void __launch_bounds__(256)
gram_part_kernel(const float* __restrict__ x, int64_t rows, int R, int64_t rows_per_block, float* __restrict__ part) {
  constexpr int RP = 16 * TR;
  __shared__ __align__(16) float xs[32][RP];    // a slab of 32 rows, zero-padded to RP columns
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  const int64_t r1 = min(rows, r0 + rows_per_block);
  float acc[TR][TR];
#pragma unroll
  for (int i = 0; i < TR; ++i)
#pragma unroll
    for (int j = 0; j < TR; ++j) acc[i][j] = 0.f;
  // a slab's 32 x RP values travel global -> registers -> shared memory; the loads of slab s + 1 are issued before slab s is
  // multiplied (a load -> store loop paid the memory latency once per element and thread: 5 of the kernel's 28 us were math)
  constexpr int PER = 32 * RP / 256;
  float pre[PER];
  auto fetch = [&](int64_t base) {
    const int nr = (int)min((int64_t)32, r1 - base);
#pragma unroll
    for (int m = 0; m < PER; ++m) {
      const int i = threadIdx.x + m * 256, rr = i / RP, col = i - rr * RP;
      pre[m] = (rr < nr && col < R) ? x[(base + rr) * R + col] : 0.f;
    }
  };
  if (r0 < r1) fetch(r0);
  for (int64_t base = r0; base < r1; base += 32) {
    __syncthreads();
#pragma unroll
    for (int m = 0; m < PER; ++m) {
      const int i = threadIdx.x + m * 256;
      xs[i / RP][i % RP] = pre[m];
    }
    __syncthreads();
    if (base + 32 < r1) fetch(base + 32);
#pragma unroll 4
    for (int rr = 0; rr < 32; ++rr) {            // rows in order: the same summation order per output as a plain loop
      float av[TR], bv[TR];
#pragma unroll
      for (int i = 0; i < TR; ++i) av[i] = xs[rr][ty * TR + i];
#pragma unroll
      for (int j = 0; j < TR; j += 4) {
        const float4 t = *reinterpret_cast<const float4*>(&xs[rr][tx * TR + j]);
        bv[j] = t.x; bv[j + 1] = t.y; bv[j + 2] = t.z; bv[j + 3] = t.w;
      }
#pragma unroll
      for (int i = 0; i < TR; ++i)
#pragma unroll
        for (int j = 0; j < TR; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
  }
  const int nout = R * R;
#pragma unroll
  for (int i = 0; i < TR; ++i)
#pragma unroll
    for (int j = 0; j < TR; ++j) {
      const int gi = ty * TR + i, gj = tx * TR + j;
      if (gi < R && gj < R) part[(int64_t)blockIdx.x * nout + gi * R + gj] = acc[i][j];
    }
}
// out[o] = sum over the nb slabs, fixed order: warp w of a block sums slabs w, w + 8, ... of 32 outputs, then the eight
// slice sums are added in order (one thread per output walking all slabs serially took 20 us for 256 slabs)
__global__ void __launch_bounds__(256)
gram_sum_kernel(const float* __restrict__ part, int nb, int nout, float* __restrict__ out) {
  __shared__ float red[8][32];
  const int lane = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const int o = blockIdx.x * 32 + lane;
  float t = 0.f;
  if (o < nout) {
#pragma unroll 4
    for (int b = sl; b < nb; b += 8) t += part[(int64_t)b * nout + o];
  }
  red[sl][lane] = t;
  __syncthreads();
  if (sl == 0 && o < nout) {
    float u = red[0][lane];
#pragma unroll
    for (int k = 1; k < 8; ++k) u += red[k][lane];
    out[o] = u;
  }
}

// Row tiles of 64: thread (ty, tx) owns rows 4 ty .. 4 ty + 3 and components TR tx .. TR tx + TR - 1 of the tile.  The tile's
// old values are staged before anything is overwritten (pitch RP + 1: the four rows of a thread and the two row groups of a
// warp fall into different banks), the Gram matrix once per block.  Dynamic shared memory: gram RP x RP | tile 64 x (RP + 1).
template <int TR>
__global__ void __launch_bounds__(256, TR == 4 ? 3 : 1)
tc_apply_eu_kernel(TcApplyArgs a, const float* __restrict__ gram) {
  constexpr int RP = 16 * TR, FP = RP + 1;
  extern __shared__ __align__(16) float eu_smem[];
  float* gs = eu_smem;                           // [RP][RP], zero-padded
  float* fs = eu_smem + RP * RP;                 // [64][FP]
  __shared__ float red[16][RP];
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
  const int64_t row0 = (int64_t)blockIdx.x * a.rpb;
  const int64_t row1 = min(a.rows, row0 + a.rpb);
  const int R = a.R;
  // staging: sixteen independent loads in flight per thread, then the stores (see gram_part_kernel)
  for (int i0 = threadIdx.x; i0 < RP * RP; i0 += 256 * 16) {
    float t[16];
#pragma unroll
    for (int m = 0; m < 16; ++m) {
      const int i = i0 + m * 256, k = i / RP, r = i - k * RP;
      t[m] = (k < R && r < R) ? gram[k * R + r] : 0.f;
    }
#pragma unroll
    for (int m = 0; m < 16; ++m) gs[i0 + m * 256] = t[m];
  }
  float cs[TR], mx = 0.f;
#pragma unroll
  for (int j = 0; j < TR; ++j) cs[j] = 0.f;
  const float kap = *a.kappa;
  for (int64_t base = row0; base < row1; base += 64) {
    __syncthreads();                             // gram staged / the previous tile's reads are done
    for (int i0 = threadIdx.x; i0 < 64 * RP; i0 += 256 * 16) {
      float t[16];
#pragma unroll
      for (int m = 0; m < 16; ++m) {
        const int i = i0 + m * 256, rl = i / RP, k = i - rl * RP;
        const int64_t row = base + rl;
        t[m] = (row < row1 && k < R) ? a.param[row * R + k] : 0.f;
      }
#pragma unroll
      for (int m = 0; m < 16; ++m) {
        const int i = i0 + m * 256;
        fs[(i / RP) * FP + (i % RP)] = t[m];
      }
    }
    // this thread's partial numerators (chunk sums, 16-byte loads; the partial rows are Rp = RP floats wide): issued before
    // the product below so that their latency hides behind it
    float numv[4][TR];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < TR; ++j) numv[i][j] = 0.f;
    for (int ch = 0; ch < a.nchunks; ++ch) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int64_t row = base + ty * 4 + i;
        if (row < row1) {
#pragma unroll
          for (int j = 0; j < TR; j += 4) {
            const float4 t = *reinterpret_cast<const float4*>(a.num + ch * a.chunk_stride + row * a.Rp + tx * TR + j);
            numv[i][j] += t.x; numv[i][j + 1] += t.y; numv[i][j + 2] += t.z; numv[i][j + 3] += t.w;
          }
        }
      }
    }
    __syncthreads();
    float acc[4][TR];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < TR; ++j) acc[i][j] = 0.f;
#pragma unroll 4
    for (int k = 0; k < RP; ++k) {               // (F G^T G)[row, r] = S^T-contraction, nmf.py:82; k ascending
      float fv[4], gv[TR];
#pragma unroll
      for (int i = 0; i < 4; ++i) fv[i] = fs[(ty * 4 + i) * FP + k];
#pragma unroll
      for (int j = 0; j < TR; j += 4) {
        const float4 t = *reinterpret_cast<const float4*>(&gs[k * RP + tx * TR + j]);
        gv[j] = t.x; gv[j + 1] = t.y; gv[j + 2] = t.z; gv[j + 3] = t.w;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < TR; ++j) acc[i][j] = fmaf(fv[i], gv[j], acc[i][j]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int64_t row = base + ty * 4 + i;
      if (row >= row1) continue;
#pragma unroll
      for (int j = 0; j < TR; ++j) {
        const int r = tx * TR + j;
        if (r >= R) continue;
        const float den = acc[i][j];
        const float num = fmaf(kap, den, numv[i][j]);            // numerator = (V - kappa S) G + kappa S G
        const float v = mu_step(fs[(ty * 4 + i) * FP + r], num, fmaxf(den, 0.f) + kEps, a.l1, a.l2, a.gamma);   // nmf.py:83
        a.param[row * R + r] = v;
        cs[j] += v;
        mx = fmaxf(mx, v);
      }
    }
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < TR; ++j) red[ty][tx * TR + j] = cs[j];
  __syncthreads();
  if (threadIdx.x < R) {
    float t = 0.f;
    for (int k = 0; k < 16; ++k) t += red[k][threadIdx.x];
    a.cs_part[(int64_t)blockIdx.x * 128 + threadIdx.x] = t;
  }
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0 && mx > 0.f) atomicMax(a.absmax, __float_as_uint(mx));
}

// fp32 factor (rows x R) -> fp16 operand copy (rows x KW): [hi(0..Rp) | lo(Rp..2Rp)] scaled by 2^a, a from the
// max found by tc_apply_kernel; pad columns stay zero (buffer zero-initialised once).  Block 0 additionally
// finishes the column sums, publishes exps[1 + which] = a, and re-derives kappa = sum(V) / sum(W H^T) =
// sum(V) / <colsum W, colsum H> (the typical P = V / (WH)) and the ratio-tile exponent exps[3] with kappa 2^p in [1, 2).
template <bool SPLIT>
__global__ void __launch_bounds__(256)
tc_finish_kernel(const float* __restrict__ x, int64_t rows, int R, __half* __restrict__ out, int KW, int Rp,
                 const unsigned int* __restrict__ absmax, unsigned int* __restrict__ absmax_next,
                 int* __restrict__ exps, int which, const float* __restrict__ cs_part, int cs_blocks,
                 float* __restrict__ colsum /* [2][R] */, const double* __restrict__ vconst,
                 float* __restrict__ kappa, int center, float* __restrict__ cs_super, unsigned int* __restrict__ ticket,
                 float bm1, float bm2, double cells) {
  const int a = pow2_exp_for(__uint_as_float(*absmax));
  const float sc = exp2f((float)a);
  if ((R & 7) == 0) {
    // 8 consecutive rank lanes per thread: two float4 loads, one 16-byte store per half
    const int per_row = R >> 3;
    const int64_t g = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (g < rows * per_row) {
      const int64_t row = g / per_row;
      const int r8 = (int)(g - row * per_row) * 8;
      const float4 a0 = *reinterpret_cast<const float4*>(x + row * R + r8);
      const float4 a1 = *reinterpret_cast<const float4*>(x + row * R + r8 + 4);
      const float xv[8] = {a0.x * sc, a0.y * sc, a0.z * sc, a0.w * sc, a1.x * sc, a1.y * sc, a1.z * sc, a1.w * sc};
      __half2 hi[4], lo[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        hi[i] = __floats2half2_rn(xv[2 * i], xv[2 * i + 1]);
        const float2 hf = __half22float2(hi[i]);
        lo[i] = __floats2half2_rn(xv[2 * i] - hf.x, xv[2 * i + 1] - hf.y);
      }
      *reinterpret_cast<uint4*>(out + row * KW + r8) = *reinterpret_cast<const uint4*>(hi);
      if (SPLIT) *reinterpret_cast<uint4*>(out + row * KW + Rp + r8) = *reinterpret_cast<const uint4*>(lo);
    }
  } else {
    for (int64_t idx = (int64_t)blockIdx.x * 256 + threadIdx.x; idx < rows * R; idx += (int64_t)gridDim.x * 256) {
      const int64_t row = idx / R;
      const int r = (int)(idx - row * R);
      const float xs = x[idx] * sc;
      const __half hi = __float2half_rn(xs);
      out[row * KW + r] = hi;
      if (SPLIT) out[row * KW + Rp + r] = __float2half_rn(xs - __half2float(hi));
    }
  }
  // ---- column sums: fixed-order two-level tree.  Blocks 0..nsuper-1 each fold a slab of the per-block partials
  // written by tc_apply_kernel; the last of them to finish (ticket counter) folds the nsuper slab sums and publishes
  // colsum, the operand exponent, kappa and the ratio-tile exponent.  The result does not depend on which block is last.
  const int nsuper = min((int)gridDim.x, 32);
  if ((int)blockIdx.x < nsuper) {
    __shared__ float partg[256];
    __shared__ int s_last;
    const int lanes = R <= 32 ? 32 : (R <= 64 ? 64 : 128);
    const int groups = 256 / lanes;
    const int r = threadIdx.x % lanes, g = threadIdx.x / lanes;
    const int per = (cs_blocks + nsuper - 1) / nsuper;
    const int b0 = blockIdx.x * per, b1 = min(cs_blocks, b0 + per);
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    int b = b0 + g;
    for (; b + 3 * groups < b1; b += 4 * groups) {
#pragma unroll
      for (int k = 0; k < 4; ++k) acc[k] += cs_part[(int64_t)(b + k * groups) * 128 + r];
    }
    for (; b < b1; b += groups) acc[0] += cs_part[(int64_t)b * 128 + r];
    partg[threadIdx.x] = (acc[0] + acc[1]) + (acc[2] + acc[3]);
    __syncthreads();
    if (threadIdx.x < lanes) {
      float mine = 0.f;
      for (int k = 0; k < groups; ++k) mine += partg[k * lanes + threadIdx.x];
      cs_super[(int64_t)blockIdx.x * 128 + threadIdx.x] = mine;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(ticket, 1u) == (unsigned)(nsuper - 1)) ? 1 : 0;
    __syncthreads();
    if (s_last) {
      __shared__ float prod[128];
      __threadfence();
      if (threadIdx.x < 128) {
        float mine = 0.f;
        if (threadIdx.x < lanes)
          for (int k = 0; k < nsuper; ++k) mine += cs_super[(int64_t)k * 128 + threadIdx.x];
        if (threadIdx.x < R) colsum[which * R + threadIdx.x] = mine;
        prod[threadIdx.x] = threadIdx.x < R ? mine * colsum[(1 - which) * R + threadIdx.x] : 0.f;
      }
      __syncthreads();
      if (threadIdx.x == 0) {
        *ticket = 0u;
        float dot = 0.f;
        for (int k = 0; k < 128; ++k) dot += prod[k];
        publish_scales(a, which, exps, absmax_next, dot, vconst, kappa, center, bm1, bm2, cells);
      }
    }
  }
}

// ---- ratio stage + operand refresh in ONE cooperative kernel (R % 4 == 0; beta != 2) ------------------------------------
// Phase 1 = the ratio stage of tc_apply_kernel with one thread per four consecutive rank lanes (nmf.py:78-92 in place,
// per-block column sums, global max); grid barrier; phase 2 = the
// fp16 operand copy with the exponent from that max (rows re-read from L2), while block 0 folds the column sums in fixed
// order and publishes colsum / kappa / exponents.  Replaces two launches, one pass over the factor and the ticket
// protocol of tc_finish_kernel; the W side also gets 2 x #SM blocks instead of rows / 64.
struct TcFinishArgs {
  __half* out; int KW, Rp;
  unsigned int* absmax; unsigned int* absmax_next;
  int* exps; int which;
  float* colsum; const double* vconst; float* kappa; int center;
  float bm1, bm2; double cells;
};

// sum over the chunked partial slabs of one float4, four independent loads in flight, fixed summation order
__device__ __forceinline__ float4 sum_chunks4(const float* __restrict__ p, int nchunks, int64_t stride) {
  float4 acc[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  int ch = 0;
  for (; ch + 4 <= nchunks; ch += 4) {
    float4 t[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) t[k] = __ldcs(reinterpret_cast<const float4*>(p + (int64_t)(ch + k) * stride));
#pragma unroll
    for (int k = 0; k < 4; ++k) { acc[k].x += t[k].x; acc[k].y += t[k].y; acc[k].z += t[k].z; acc[k].w += t[k].w; }
  }
  for (; ch < nchunks; ++ch) {
    const float4 t = __ldcs(reinterpret_cast<const float4*>(p + (int64_t)ch * stride));
    acc[0].x += t.x; acc[0].y += t.y; acc[0].z += t.z; acc[0].w += t.w;
  }
  return make_float4((acc[0].x + acc[1].x) + (acc[2].x + acc[3].x), (acc[0].y + acc[1].y) + (acc[2].y + acc[3].y),
                     (acc[0].z + acc[1].z) + (acc[2].z + acc[3].z), (acc[0].w + acc[1].w) + (acc[2].w + acc[3].w));
}

// the same float4 of every rank's packed buffer (slots of THIS rank's exchange block, written by their owners over NVLink),
// summed in rank order: identical on every rank.  L2 loads: remote writes land in this GPU's L2, never in an SM's L1.
__device__ __forceinline__ float4 sum_peers4(const float* const* peers, int npeers, int64_t off) {
  float4 t[kMaxPeers];
#pragma unroll
  for (int p = 0; p < kMaxPeers; ++p)
    if (p < npeers) t[p] = __ldcg(reinterpret_cast<const float4*>(peers[p] + off));
  float4 acc = t[0];
#pragma unroll
  for (int p = 1; p < kMaxPeers; ++p)
    if (p < npeers) { acc.x += t[p].x; acc.y += t[p].y; acc.z += t[p].z; acc.w += t[p].w; }
  return acc;
}

// one rank's "buffer published" counters, written by the peers over NVLink; bounded wait (a rank that never arrives must not
// hang the GPU: the error word is checked by the host's health check)
__device__ __forceinline__ void wait_peer_flags(const unsigned int* flags, int npeers, unsigned int target, unsigned int* err) {
  if ((int)threadIdx.x < npeers) {
    const long long t0 = clock64();
    unsigned int v;
    for (;;) {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + threadIdx.x) : "memory");
      if ((int)(v - target) >= 0) break;
      if (clock64() - t0 > 4000000000LL) { atomicExch(err, 1u + threadIdx.x); break; }
    }
  }
  __syncthreads();
}

template <bool SPLIT>
__global__ void __launch_bounds__(256)
tc_apply_finish_kernel(TcApplyArgs a, TcFinishArgs f) {
  __shared__ float4 sh[256];
  const int lanes = a.R >> 2;                    // threads per row
  const int rows_per_pass = 256 / lanes;
  const int rl = threadIdx.x / lanes, q = threadIdx.x - rl * lanes;      // row slot, rank quad
  const int64_t row0 = (int64_t)blockIdx.x * a.rpb;
  const int64_t row1 = min(a.rows, row0 + a.rpb);
  float4 cs = make_float4(0.f, 0.f, 0.f, 0.f);
  float mx = 0.f;
  const bool peer = a.npeers > 0;
  if (peer) wait_peer_flags(a.flags, a.npeers, a.flag_target, a.peer_err);
  const int64_t RR = a.rows * a.R;               // peer buffers: [rows x R | colsum R (beta 1) or rows x R]
  if (rl < rows_per_pass) {
    float4 kd = make_float4(1.f, 1.f, 1.f, 1.f);
    float kap = 0.f;
    if (a.apply && !a.den) {
      kd = peer ? sum_peers4(a.peers, a.npeers, RR + 4 * q) : *reinterpret_cast<const float4*>(a.kl_den + 4 * q);
      kap = *a.kappa;
    }
    for (int64_t row = row0 + rl; row < row1; row += rows_per_pass) {
      float4* pp = reinterpret_cast<float4*>(a.param + row * a.R) + q;
      float4 v = *pp;
      if (a.apply) {
        const float4 num = peer ? sum_peers4(a.peers, a.npeers, row * a.R + 4 * q)
                                : sum_chunks4(a.num + row * a.Rp + 4 * q, a.nchunks, a.chunk_stride);
        const float4 dsum = !a.den ? make_float4(0.f, 0.f, 0.f, 0.f)
                            : peer ? sum_peers4(a.peers, a.npeers, RR + row * a.R + 4 * q)
                                   : sum_chunks4(a.den + row * a.Rp + 4 * q, a.nchunks, a.chunk_stride);
        float vv[4] = {v.x, v.y, v.z, v.w}, nn[4] = {num.x, num.y, num.z, num.w}, dd[4] = {kd.x, kd.y, kd.z, kd.w};
        const float ds[4] = {dsum.x, dsum.y, dsum.z, dsum.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float n = a.den ? nn[i] : fmaf(kap, dd[i], nn[i]);  // beta == 1: the kernel accumulated sum (P - kappa) G
          const float pos = a.den ? fmaxf(ds[i], 0.f) + kEps : dd[i];   // nmf.py:83 | nmf.py:368-369 / :381-382
          vv[i] = mu_step(vv[i], n, pos, a.l1, a.l2, a.gamma);
        }
        v = make_float4(vv[0], vv[1], vv[2], vv[3]);
        *pp = v;
      }
      cs.x += v.x; cs.y += v.y; cs.z += v.z; cs.w += v.w;
      mx = fmaxf(fmaxf(mx, fmaxf(v.x, v.y)), fmaxf(v.z, v.w));
    }
  }
  sh[threadIdx.x] = cs;
  __syncthreads();
  if (threadIdx.x < lanes) {
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int k = 0; k < rows_per_pass; ++k) {
      const float4 u = sh[k * lanes + threadIdx.x];
      t.x += u.x; t.y += u.y; t.z += u.z; t.w += u.w;
    }
    *(reinterpret_cast<float4*>(a.cs_part + (int64_t)blockIdx.x * 128) + threadIdx.x) = t;
  }
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0 && mx > 0.f) atomicMax(f.absmax, __float_as_uint(mx));
  __threadfence();
  cooperative_groups::this_grid().sync();

  // ---- phase 2: fp16 operand copy of this block's rows (just written: L2 hits), scaled by 2^a from the global max
  const int ae = pow2_exp_for(__uint_as_float(*reinterpret_cast<volatile unsigned int*>(f.absmax)));
  const float sc = exp2f((float)ae);
  if (rl < rows_per_pass) {
    for (int64_t row = row0 + rl; row < row1; row += rows_per_pass) {
      const float4 v = __ldcg(reinterpret_cast<const float4*>(a.param + row * a.R) + q);
      const float xv[4] = {v.x * sc, v.y * sc, v.z * sc, v.w * sc};
      __half2 hi[2], lo[2];
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        hi[i] = __floats2half2_rn(xv[2 * i], xv[2 * i + 1]);
        const float2 hf = __half22float2(hi[i]);
        lo[i] = __floats2half2_rn(xv[2 * i] - hf.x, xv[2 * i + 1] - hf.y);
      }
      *reinterpret_cast<uint2*>(f.out + row * f.KW + 4 * q) = *reinterpret_cast<const uint2*>(hi);
      if (SPLIT) *reinterpret_cast<uint2*>(f.out + row * f.KW + f.Rp + 4 * q) = *reinterpret_cast<const uint2*>(lo);
    }
  }
  // ---- block 0: column sums in fixed order (two halves of the block list, then their sum), then the scalars
  if (blockIdx.x == 0) {
    __shared__ float partg[256];
    __shared__ float prod[128];
    const int fl = a.R <= 32 ? 32 : (a.R <= 64 ? 64 : 128);     // lanes per group; 256 / fl groups walk the block list
    const int groups = 256 / fl;
    const int r = threadIdx.x % fl, g = threadIdx.x / fl;
    // this one block is on the kernel's critical path: 16 loads in flight per thread (an L2 round trip per batch)
    float acc16[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) acc16[k] = 0.f;
    if (r < a.R) {
      int b = g;
      for (; b + 15 * groups < (int)gridDim.x; b += 16 * groups) {
        float t[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) t[k] = __ldcg(a.cs_part + (int64_t)(b + k * groups) * 128 + r);
#pragma unroll
        for (int k = 0; k < 16; ++k) acc16[k] += t[k];
      }
      for (; b < (int)gridDim.x; b += groups) acc16[0] += __ldcg(a.cs_part + (int64_t)b * 128 + r);
    }
    float accs = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k) accs += acc16[k];
    partg[threadIdx.x] = accs;
    __syncthreads();
    if (threadIdx.x < 128) {
      float mine = 0.f;
      if (threadIdx.x < fl)
        for (int k = 0; k < groups; ++k) mine += partg[k * fl + threadIdx.x];
      if (threadIdx.x < a.R) f.colsum[f.which * a.R + threadIdx.x] = mine;
      prod[threadIdx.x] = threadIdx.x < a.R ? mine * f.colsum[(1 - f.which) * a.R + threadIdx.x] : 0.f;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      float dot = 0.f;
      for (int k = 0; k < 128; ++k) dot += prod[k];
      publish_scales(ae, f.which, f.exps, f.absmax_next, dot, f.vconst, f.kappa, f.center, f.bm1, f.bm2, f.cells);
    }
  }
}

struct PeerSignal { unsigned int* ticket; unsigned int* const* peer_flags; int world, rank; unsigned int iter; };

// Peer-memory W update, producer side: this rank's packed partial [rows x R | colsum R (beta 1) or rows x R] is PUSHED into
// slot `rank` of every rank's exchange block (posted NVLink writes; P2P reads of the same data measured 10x slower), then the
// block that finishes last publishes this rank's iteration counter into every rank's flag array.
struct PeerPush { float* dst[kMaxPeers]; };

__global__ void __launch_bounds__(256)
w_pack_push_kernel(const float* __restrict__ num, const float* __restrict__ den, int nchunks, int64_t chunk_stride,
                   int64_t rows, int R, int Rp, const float* __restrict__ colsum_h, const float* __restrict__ kappa,
                   PeerPush out, PeerSignal sig) {
  const int64_t CR = rows * R, total = den ? 2 * CR : CR + R;
  const int64_t i = ((int64_t)blockIdx.x * 256 + threadIdx.x) * 4;      // R % 4 == 0: four elements of one row
  if (i < total) {
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < CR || den) {
      const bool second = i >= CR;
      const int64_t j = second ? i - CR : i;
      const int64_t row = j / R;
      const int r = (int)(j - row * R);
      const float* src = (second ? den : num) + row * Rp + r;
      for (int ch = 0; ch < nchunks; ++ch) {
        const float4 t = *reinterpret_cast<const float4*>(src + ch * chunk_stride);
        a.x += t.x; a.y += t.y; a.z += t.z; a.w += t.w;
      }
      if (!den) {
        const float k = *kappa;
        const float4 c = *reinterpret_cast<const float4*>(colsum_h + r);
        a.x = fmaf(k, c.x, a.x); a.y = fmaf(k, c.y, a.y); a.z = fmaf(k, c.z, a.z); a.w = fmaf(k, c.w, a.w);
      }
    } else {
      a = *reinterpret_cast<const float4*>(colsum_h + (i - CR));
    }
#pragma unroll
    for (int p = 0; p < kMaxPeers; ++p)
      if (p < sig.world) *reinterpret_cast<float4*>(out.dst[p] + i) = a;
  }
  __shared__ int last;
  __threadfence_system();                 // this thread's remote writes are performed before the ticket below
  __syncthreads();
  if (threadIdx.x == 0) {
    last = atomicAdd(sig.ticket, 1u) == gridDim.x - 1;
    if (last) *sig.ticket = 0u;
  }
  __syncthreads();
  if (last && (int)threadIdx.x < sig.world) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(sig.peer_flags[threadIdx.x] + sig.rank), "r"(sig.iter) : "memory");
  }
}

// Row-sharded W update: this rank's contribution to the all-reduce buffer in one pass (was: chunk reduction, D2D copy,
// row-vector add).  den == nullptr (beta 1): out = [num + kappa colsum_h | colsum_h]; otherwise out = [num | den].
__global__ void __launch_bounds__(256)
w_partial_pack_kernel(const float* __restrict__ num, const float* __restrict__ den, int nchunks, int64_t chunk_stride,
                      int64_t rows, int R, int Rp, const float* __restrict__ colsum_h, const float* __restrict__ kappa,
                      float* __restrict__ out) {
  const int64_t CR = rows * R;
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i < CR) {
    const int64_t row = i / R;
    const int r = (int)(i - row * R);
    const int64_t off = row * Rp + r;
    float a = 0.f;
    for (int ch = 0; ch < nchunks; ++ch) a += num[ch * chunk_stride + off];
    out[i] = den ? a : fmaf(*kappa, colsum_h[r], a);
  } else if (den) {
    if (i < 2 * CR) {
      const int64_t j = i - CR;
      const int64_t row = j / R;
      const int r = (int)(j - row * R);
      float a = 0.f;
      for (int ch = 0; ch < nchunks; ++ch) a += den[ch * chunk_stride + row * Rp + r];
      out[i] = a;
    }
  } else if (i < CR + R) {
    out[i] = colsum_h[i - CR];
  }
}

// loss = sum V log(V+eps) - sum V - ln2 * 2^-v * sum v~ lg2(S+eps) + 2^-(aW+aH) * sum S~      (metrics.py:22)
__global__ void tc_loss_final_kernel(const double* __restrict__ part, int nblk, const double* __restrict__ vconst,
                                     const int* __restrict__ exps, double* __restrict__ out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double a = 0.0, b = 0.0;
  for (int i = 0; i < nblk; ++i) { a += part[2 * i]; b += part[2 * i + 1]; }
  const double ln2 = 0.693147180559945309417;
  *out = vconst[1] - vconst[0] - ln2 * exp2((double)-exps[0]) * a + exp2((double)-(exps[1] + exps[2])) * b;
}

// beta != 1 (metrics.py:56-57, :84-96): vb = the V-only term for this beta (sum ln(V+eps) or sum t^beta)
__global__ void tc_loss_final_beta_kernel(const double* __restrict__ part, int nblk, const double* __restrict__ vb,
                                          double beta, double cells, double* __restrict__ out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double a = 0.0, b = 0.0;
  for (int i = 0; i < nblk; ++i) { a += part[2 * i]; b += part[2 * i + 1]; }
  const double ln2 = 0.693147180559945309417;
  if (beta == 2.0) *out = 0.5 * a;
  else if (beta == 0.0) *out = a - *vb + ln2 * b - cells;
  else *out = (*vb + (beta - 1.0) * b - beta * a) / (beta * (beta - 1.0));
}

// V-only loss term: beta == 0: sum ln(V + eps); else sum t^beta with t = V (+ eps if beta < 0).  Two-level, fixed order.
__global__ void __launch_bounds__(256)
v_beta_term_kernel(const float* __restrict__ V, int64_t rows, int64_t cols, int64_t ld, float beta,
                   double* __restrict__ blockpart) {
  __shared__ double red[8];
  double acc = 0.0;
  const int64_t total = rows * cols;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < total; i += (int64_t)gridDim.x * 256) {
    const int64_t r = i / cols, c = i - r * cols;
    const float v = V[r * ld + c];
    acc += (double)(beta == 0.f ? logf(v + kEps) : powf(beta < 0.f ? v + kEps : v, beta));
  }
  const double t = block_sum256(acc, red);
  if (threadIdx.x == 0) blockpart[blockIdx.x] = t;
}
__global__ void __launch_bounds__(256)
sum_blocks_kernel(const double* __restrict__ blockpart, int n, double* __restrict__ out) {
  __shared__ double red[8];
  double acc = 0.0;
  for (int i = threadIdx.x; i < n; i += 256) acc += blockpart[i];
  const double t = block_sum256(acc, red);
  if (threadIdx.x == 0) *out = t;
}

// ---- host side --------------------------------------------------------------------------------------

struct Plan { int row_blocks, tiles, nchunks, tpc; };

Plan make_plan(int64_t Mr, int64_t Nc, int num_sms, int TN) {
  Plan pl;
  pl.row_blocks = (int)ceil_div(Mr, kTileM);
  pl.tiles = (int)ceil_div(Nc, TN);
  int best = 1;
  double best_eff = -1.0;
  for (int nch = 1; nch <= pl.tiles && nch <= 64; ++nch) {
    int tpc = (int)ceil_div(pl.tiles, nch);
    if (tpc * TN < 512 && nch > 1) break;
    int real = (int)ceil_div(pl.tiles, tpc);
    if (real != nch) continue;
    int64_t items = (int64_t)pl.row_blocks * nch;
    double eff = (double)items / (double)(ceil_div(items, num_sms) * num_sms);
    // fewer chunks = less partial traffic: only move on for a clear win
    if (eff > best_eff + 0.03) { best_eff = eff; best = nch; }
    if (best_eff >= 0.97) break;
  }
  pl.nchunks = best;
  pl.tpc = (int)ceil_div(pl.tiles, best);
  return pl;
}

}  // namespace

static PFN_cuTensorMapEncodeTiled_v12000 get_encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (fn) return fn;
  void* ptr = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(ptr);
  return fn;
}

int make_tmap(CUtensorMap* m, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
  auto fn = get_encode_fn();
  if (!fn) { set_error("cuTensorMapEncodeTiled entry point not available"); return 2; }
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with code " + std::to_string((int)r)); return 2; }
  return 0;
}

struct TcState {
  // ---- row-sharded W update over peer memory (tc_peer_*): one cudaMalloc block per rank, shared by CUDA IPC:
  //      [64 counters: flags[p] = last iteration rank p published][parity 0: 8 slots][parity 1: 8 slots]; slot p of every
  //      block is written by rank p (2 C R floats each)
  void* peer_block = nullptr;                    // this rank's block
  void* peer_base[kMaxPeers] = {};               // every rank's block in this process' address space (own: peer_block)
  unsigned int** peer_flag_tab = nullptr;        // device copy of the flag-array pointers (for the signal kernel)
  unsigned int* peer_err = nullptr;
  int peer_world = 0, peer_rank = 0;
  unsigned int peer_iter = 0;
  int64_t peer_buf_floats = 0;
  int device = 0, num_sms = 148;
  int64_t N = 0, C = 0, R = 0;
  bool split = true;
  int Rp = 64;                      // padded rank: 64 or 128
  int TN = 128;                     // tile width of the contraction kernel for this (Rp, split)
  int KW = 128;
  int64_t ldc = 0, ldn = 0;
  __half *V16 = nullptr, *Vt16 = nullptr, *W16 = nullptr, *H16 = nullptr;
  float* part = nullptr;
  float* part2 = nullptr;           // denominators of the beta != 1 kernels (allocated on first use)
  float* gram = nullptr;            // beta 2: G^T G (R x R) and its per-slab partials [256][R*R] (allocated on first use)
  float* gram_part = nullptr;
  int64_t part_floats = 0;
  float* colsum = nullptr;          // [2][R]  0 = W, 1 = H
  float* cs_part = nullptr;         // [<=1024][128]
  float* cs_super = nullptr;        // [32][128]
  unsigned int* ticket = nullptr;
  unsigned int* absmax = nullptr;   // [2 factors][2 parities]
  int* exps = nullptr;              // {v, aW, aH, p}
  double* vpart = nullptr;          // per-block {sum V, sum V log V}
  int64_t vblocks = 0;
  double* vconst = nullptr;         // {sum V, sum V log(V+eps)}
  unsigned long long* vlossy = nullptr;   // positive target entries the scaled fp16 copy cannot hold at full precision
  double* loss_part = nullptr;      // [num_sms][2]
  bool w_pending = false;           // tc_loss_prefetch_w: the W update's partial numerators of the CURRENT factors are in `part`
  const float* Vsrc = nullptr;      // the registered fp32 target (borrowed) for the V-only loss terms
  int64_t ldv = 0;
  double* vbeta = nullptr;          // device: V-only loss term of beta `vbeta_for`
  double* vbeta_part = nullptr;     // [1024]
  double vbeta_for = 1.0;           // 1.0 = none cached
  CUtensorMap tmV, tmVt;            // V16 / Vt16, box 64 x 128
  CUtensorMap tmWf, tmHf;           // factors as the row factor F: box 64 x 128
  CUtensorMap tmWg, tmHg;           // factors as the column factor G: box 64 x TN
  Plan plan_w, plan_h;
  uint32_t upd[2] = {0, 0};         // per-factor update counter (selects the absmax slot)
  bool dirty_w = true, dirty_h = true, has_target = false;
  // Environment knobs, read once in tc_create: NMFB200_CENTER=0 (diagnostic: kappa centring off, see
  // tools/bias_probe.py), NMFB200_TC_CHECK=1 (watchdog check after every tc_contract_only).
  int center = 1;
  bool check_each = false;
  float* kappa = nullptr;           // device scalar
  float* zero = nullptr;            // device scalar 0 (kappa of an already complete numerator)
  int coop_blocks = 0;              // co-resident blocks of the fused tail kernel (cooperative launch), 0 = unavailable
};

bool tc_shape_supported(int64_t N, int64_t C, int64_t R) {
  // the conversion kernel walks 64-row slabs on gridDim.y (<= 65535): taller targets take the fp32 kernels
  return R >= 1 && R <= 128 && N >= 1 && C >= 1 && N <= 65535ll * 64 && C < (1ll << 31);
}

void tc_peer_release(TcState* s) {
  for (int p = 0; p < s->peer_world; ++p)
    if (p != s->peer_rank && s->peer_base[p]) cudaIpcCloseMemHandle(s->peer_base[p]);
  for (auto& b : s->peer_base) b = nullptr;
  cudaFree(s->peer_block); s->peer_block = nullptr;
  cudaFree(s->peer_flag_tab); s->peer_flag_tab = nullptr;
  cudaFree(s->peer_err); s->peer_err = nullptr;
  s->peer_world = 0; s->peer_iter = 0;
}

void tc_destroy(TcState* s) {
  if (!s) return;      // the caller (capi.cu: free_ctx) has selected s->device
  tc_peer_release(s);
  cudaFree(s->V16); cudaFree(s->Vt16); cudaFree(s->W16); cudaFree(s->H16); cudaFree(s->part); cudaFree(s->part2); cudaFree(s->gram); cudaFree(s->gram_part);
  cudaFree(s->colsum); cudaFree(s->cs_part); cudaFree(s->cs_super); cudaFree(s->ticket); cudaFree(s->absmax); cudaFree(s->exps);
  cudaFree(s->vpart); cudaFree(s->vconst); cudaFree(s->vlossy); cudaFree(s->loss_part); cudaFree(s->vbeta); cudaFree(s->vbeta_part); cudaFree(s->kappa); cudaFree(s->zero);
  delete s;
}

int tc_create(TcState** out, int device, int64_t N, int64_t C, int64_t R, bool split) {
  *out = nullptr;
  TcState* s = new TcState();
  s->device = device; s->N = N; s->C = C; s->R = R; s->split = split;
  s->Rp = R <= 64 ? 64 : 128;
  s->KW = split ? 2 * s->Rp : s->Rp;
  s->TN = (split && s->Rp == 128) ? 64 : 128;   // 64-column tiles only where 128 do not fit (measured slower: MMA issue rate)
  if (const char* e = getenv("NMFB200_CENTER")) s->center = atoi(e);
  s->check_each = getenv("NMFB200_TC_CHECK") != nullptr;
  s->ldc = round_up(C, 8);
  s->ldn = round_up(N, 8);
  cudaDeviceProp prop;
  NMF_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
  s->num_sms = prop.multiProcessorCount;
  if (prop.major != 10) { delete s; set_error("the tensor-core path needs an sm_100 device"); return 1; }
  {
    int coop = 0, per_sm = 0;
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device);
    const void* fn = split ? (const void*)tc_apply_finish_kernel<true> : (const void*)tc_apply_finish_kernel<false>;
    if (coop && cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, 256, 0) == cudaSuccess && per_sm > 0) {
      if (per_sm > 4) per_sm = 4;                            // enough loads in flight to stream the partials
      s->coop_blocks = per_sm * s->num_sms;
      if (s->coop_blocks > 1024) s->coop_blocks = 1024;      // cs_part capacity
    }
  }
  s->plan_w = make_plan(C, N, s->num_sms, s->TN);
  s->plan_h = make_plan(N, C, s->num_sms, s->TN);
  int64_t pw = (int64_t)s->plan_w.nchunks * C * s->Rp, ph = (int64_t)s->plan_h.nchunks * N * s->Rp;
  s->part_floats = pw > ph ? pw : ph;
  s->vblocks = ceil_div(C, 64) * ceil_div(N, 64);
  cudaError_t e = cudaSuccess;
  if (e == cudaSuccess) e = cudaMalloc(&s->V16, (size_t)N * s->ldc * 2);
  if (e == cudaSuccess) e = cudaMalloc(&s->Vt16, (size_t)C * s->ldn * 2);
  if (e == cudaSuccess) e = cudaMalloc(&s->W16, (size_t)C * s->KW * 2);
  if (e == cudaSuccess) e = cudaMalloc(&s->H16, (size_t)N * s->KW * 2);
  if (e == cudaSuccess) e = cudaMalloc(&s->part, (size_t)s->part_floats * 4);
  if (e == cudaSuccess) e = cudaMalloc(&s->colsum, 2 * R * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&s->cs_part, 1024 * 128 * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&s->cs_super, 32 * 128 * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&s->ticket, sizeof(unsigned int));
  if (e == cudaSuccess) e = cudaMemset(s->ticket, 0, sizeof(unsigned int));
  if (e == cudaSuccess) e = cudaMalloc(&s->absmax, 4 * sizeof(unsigned int));
  if (e == cudaSuccess) e = cudaMalloc(&s->exps, 8 * sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc(&s->vpart, (size_t)s->vblocks * 2 * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&s->vconst, 2 * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&s->vlossy, sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaMalloc(&s->loss_part, (size_t)s->num_sms * 2 * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&s->kappa, sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&s->zero, sizeof(float));
  if (e == cudaSuccess) e = cudaMemset(s->zero, 0, sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&s->vbeta, sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&s->vbeta_part, 1024 * sizeof(double));
  if (e == cudaSuccess) e = cudaMemset(s->kappa, 0, sizeof(float));
  if (e == cudaSuccess) e = cudaMemset(s->W16, 0, (size_t)C * s->KW * 2);
  if (e == cudaSuccess) e = cudaMemset(s->H16, 0, (size_t)N * s->KW * 2);
  if (e == cudaSuccess) e = cudaMemset(s->exps, 0, 8 * sizeof(int));
  if (e == cudaSuccess) e = cudaMemset(s->absmax, 0, 4 * sizeof(unsigned int));
  if (e == cudaSuccess) e = cudaMemset(s->colsum, 0, 2 * R * sizeof(float));
  if (e == cudaSuccess) e = cudaMemset(s->vconst, 0, 2 * sizeof(double));
  if (e != cudaSuccess) {
    tc_destroy(s);
    set_error(std::string("tc_create cudaMalloc: ") + cudaGetErrorString(e));
    return 2;
  }
  int rc = 0;
  rc |= make_tmap(&s->tmV, s->V16, N, C, s->ldc, kTileM);
  rc |= make_tmap(&s->tmVt, s->Vt16, C, N, s->ldn, kTileM);
  rc |= make_tmap(&s->tmWf, s->W16, C, s->KW, s->KW, kTileM);
  rc |= make_tmap(&s->tmHf, s->H16, N, s->KW, s->KW, kTileM);
  rc |= make_tmap(&s->tmWg, s->W16, C, s->KW, s->KW, s->TN);
  rc |= make_tmap(&s->tmHg, s->H16, N, s->KW, s->KW, s->TN);
  if (rc) { tc_destroy(s); return 2; }
  *out = s;
  return 0;
}

bool tc_supports_beta(const TcState* s, double beta) {
  if (beta == 1.0) return true;
  if (beta == 2.0) return true;    // residual kernel, any configuration
  // other beta: two-output kernel (rank <= 64)
  return s->Rp == 64 && s->TN == 128;
}
bool tc_supports_partial(const TcState* s, double beta) { return beta != 2.0 && tc_supports_beta(s, beta); }

int tc_set_target(TcState* s, const float* V, int64_t ldv, const float* minmax_dev, cudaStream_t st) {
  s->w_pending = false;
  set_vexp_kernel<<<1, 32, 0, st>>>(minmax_dev, s->exps);
  NMF_LAUNCH_CHECK();
  dim3 grid((unsigned)ceil_div(s->C, 64), (unsigned)ceil_div(s->N, 64));
  NMF_CUDA_CHECK(cudaMemsetAsync(s->vlossy, 0, sizeof(unsigned long long), st));
  v_to_f16_kernel<<<grid, 256, 0, st>>>(V, ldv, (int)s->N, (int)s->C, s->V16, s->ldc, s->Vt16, s->ldn, s->exps,
                                        s->vpart, s->vlossy);
  NMF_LAUNCH_CHECK();
  reduce_vconst_kernel<<<1, 256, 0, st>>>(s->vpart, s->vblocks, s->vconst);
  NMF_LAUNCH_CHECK();
  s->has_target = true;
  s->Vsrc = V; s->ldv = ldv; s->vbeta_for = 1.0;
  s->dirty_w = s->dirty_h = true;      // exps[3] depends on sum(V)
  return 0;
}

int tc_target_lossy(TcState* s, unsigned long long* count, cudaStream_t st) {
  NMF_CUDA_CHECK(cudaMemcpyAsync(count, s->vlossy, sizeof(*count), cudaMemcpyDeviceToHost, st));
  NMF_CUDA_CHECK(cudaStreamSynchronize(st));
  return 0;
}

int tc_target_sum(TcState* s, double* vsum, cudaStream_t st) {
  NMF_CUDA_CHECK(cudaMemcpyAsync(vsum, s->vconst, sizeof(double), cudaMemcpyDeviceToHost, st));
  NMF_CUDA_CHECK(cudaStreamSynchronize(st));
  return 0;
}

void tc_mark_dirty(TcState* s, bool w, bool h) {
  if (w) s->dirty_w = true;
  if (h) s->dirty_h = true;
}

namespace {

// ratio stage (apply != 0) or plain re-scan (apply == 0) of one factor, then rebuild its fp16 operand copy,
// column sums and the exponents that depend on it: two launches.
// `reduced` != nullptr: the sharded path -- numerator (and KL denominator / raw denominator) come from the all-reduced
// buffer [rows*R num | R colsum or rows*R den] instead of this rank's chunked partials.
int apply_and_finish(TcState* s, int which, float* param, bool apply, const Plan* pl, double beta, double gamma,
                     double l1, double l2, cudaStream_t st, const float* reduced = nullptr,
                     const float* other = nullptr, bool peer = false) {
  const int64_t rows = which == 0 ? s->C : s->N;
  int rpb = (int)round_up(ceil_div(rows, 1024), 4);
  if (rpb < 64) rpb = 64;
  const int blocks = (int)ceil_div(rows, rpb);
  const uint32_t k = s->upd[which]++;
  unsigned int* slot = s->absmax + which * 2 + (k & 1);
  unsigned int* next = s->absmax + which * 2 + ((k + 1) & 1);
  TcApplyArgs a{};
  a.param = param; a.rows = rows; a.R = (int)s->R; a.rpb = rpb;
  a.num = s->part; a.nchunks = pl ? pl->nchunks : 0; a.chunk_stride = rows * s->Rp; a.Rp = s->Rp;
  a.kl_den = s->colsum + (1 - which) * s->R;     // W update divides by colsum(H), H update by colsum(W)
  a.den = (apply && beta != 1.0 && beta != 2.0) ? s->part2 : nullptr;
  if (reduced) {
    a.num = reduced; a.nchunks = 1; a.chunk_stride = 0; a.Rp = (int)s->R;
    a.kl_den = reduced + rows * s->R;
    a.den = beta != 1.0 ? reduced + rows * s->R : nullptr;
  }
  a.gamma = (float)gamma; a.l1 = (float)l1; a.l2 = (float)l2;
  a.cs_part = s->cs_part; a.absmax = slot; a.apply = apply ? 1 : 0; a.kappa = reduced ? s->zero : s->kappa;
  if (peer) {
    if (!((s->R & 3) == 0 && s->coop_blocks > 0)) { set_error("internal: peer W update needs the fused ratio-stage kernel"); return 1; }
    // the ranks' slots of THIS rank's block for this iteration's parity (every rank pushed its packed partial into them)
    for (int p = 0; p < s->peer_world; ++p)
      a.peers[p] = reinterpret_cast<const float*>(s->peer_block) + 64 +
                   ((int64_t)(s->peer_iter & 1u) * kMaxPeers + p) * s->peer_buf_floats;
    a.npeers = s->peer_world; a.flags = reinterpret_cast<const unsigned int*>(s->peer_block);
    a.flag_target = s->peer_iter; a.peer_err = s->peer_err;
  }
  if ((s->R & 3) == 0 && !(apply && beta == 2.0 && !reduced) && s->coop_blocks > 0) {
    // one cooperative launch: ratio stage, grid barrier, operand copy + scalars
    const int lanes = (int)s->R >> 2, rows_per_pass = 256 / lanes;
    int64_t g = ceil_div(rows, rows_per_pass);
    if (g > s->coop_blocks) g = s->coop_blocks;
    a.rpb = (int)round_up(ceil_div(rows, g), rows_per_pass);
    const int gblocks = (int)ceil_div(rows, a.rpb);
    TcFinishArgs f{};
    f.out = which == 0 ? s->W16 : s->H16; f.KW = s->KW; f.Rp = s->Rp; f.absmax = slot; f.absmax_next = next;
    f.exps = s->exps; f.which = which; f.colsum = s->colsum; f.vconst = s->vconst; f.kappa = s->kappa;
    f.center = s->center; f.bm1 = (float)(beta - 1.0); f.bm2 = (float)(beta - 2.0);
    f.cells = (double)s->N * (double)s->C;
    void* args[2] = {&a, &f};
    const void* fn = s->split ? (const void*)tc_apply_finish_kernel<true> : (const void*)tc_apply_finish_kernel<false>;
    NMF_CUDA_CHECK(cudaLaunchCooperativeKernel(fn, dim3(gblocks), dim3(256), args, 0, st));
    count_launch();
    return 0;
  }
  if (apply && beta == 2.0 && !reduced) {
    // den_raw = F (G^T G): Gram matrix of the other factor (fp32, fixed-order two-level sum), then the EU ratio stage
    if (!other) { set_error("internal: beta 2 update without the other factor"); return 1; }
    const int R = (int)s->R, nout = R * R;
    if (!s->gram) {
      NMF_CUDA_CHECK(cudaMalloc(&s->gram, (size_t)nout * 4));
      NMF_CUDA_CHECK(cudaMalloc(&s->gram_part, (size_t)256 * nout * 4));
    }
    const int64_t orows = which == 0 ? s->N : s->C;
    int64_t rpbg = round_up(ceil_div(orows, 256), 32);
    const int nb = (int)ceil_div(orows, rpbg);
    if (s->Rp == 64) gram_part_kernel<4><<<nb, 256, 0, st>>>(other, orows, R, rpbg, s->gram_part);
    else gram_part_kernel<8><<<nb, 256, 0, st>>>(other, orows, R, rpbg, s->gram_part);
    NMF_LAUNCH_CHECK();
    gram_sum_kernel<<<(unsigned)ceil_div(nout, 32), 256, 0, st>>>(s->gram_part, nb, nout, s->gram);
    NMF_LAUNCH_CHECK();
    a.den = nullptr;
    const int RPk = s->Rp == 64 ? 64 : 128;
    const int eu_smem = (RPk * RPk + 64 * (RPk + 1)) * (int)sizeof(float);
    if (RPk == 64) {
      tc_apply_eu_kernel<4><<<blocks, 256, eu_smem, st>>>(a, s->gram);
    } else {
      static unsigned long long eu_attr_mask = 0;                    // > 48 KB of dynamic shared memory: opt in once per device
      if (!((eu_attr_mask >> (s->device & 63)) & 1ull)) {
        NMF_CUDA_CHECK(cudaFuncSetAttribute(tc_apply_eu_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, eu_smem));
        eu_attr_mask |= 1ull << (s->device & 63);
      }
      tc_apply_eu_kernel<8><<<blocks, 256, eu_smem, st>>>(a, s->gram);
    }
  } else {
    tc_apply_kernel<<<blocks, 256, 0, st>>>(a);
  }
  NMF_LAUNCH_CHECK();
  __half* out = which == 0 ? s->W16 : s->H16;
  const unsigned grid = (unsigned)ceil_div((s->R & 7) == 0 ? rows * (s->R >> 3) : rows * s->R, 256);
  if (s->split)
    tc_finish_kernel<true><<<grid, 256, 0, st>>>(param, rows, (int)s->R, out, s->KW, s->Rp, slot, next, s->exps, which,
                                                 s->cs_part, blocks, s->colsum, s->vconst, s->kappa, s->center, s->cs_super, s->ticket,
                                                 (float)(beta - 1.0), (float)(beta - 2.0), (double)s->N * (double)s->C);
  else
    tc_finish_kernel<false><<<grid, 256, 0, st>>>(param, rows, (int)s->R, out, s->KW, s->Rp, slot, next, s->exps, which,
                                                  s->cs_part, blocks, s->colsum, s->vconst, s->kappa, s->center, s->cs_super, s->ticket,
                                                 (float)(beta - 1.0), (float)(beta - 2.0), (double)s->N * (double)s->C);
  NMF_LAUNCH_CHECK();
  return 0;
}

int ensure_synced(TcState* s, const float* W, const float* H, double beta, cudaStream_t st) {
  if (!s->has_target) { set_error("tensor-core path: set_target has not been called"); return 3; }
  if (s->dirty_w) {
    int rc = apply_and_finish(s, 0, const_cast<float*>(W), false, nullptr, beta, 1, 0, 0, st);
    if (rc) return rc;
    s->dirty_w = false;
  }
  if (s->dirty_h) {      // after a W refresh, this one recomputes exps[3] with both column sums valid
    int rc = apply_and_finish(s, 1, const_cast<float*>(H), false, nullptr, beta, 1, 0, 0, st);
    if (rc) return rc;
    s->dirty_h = false;
  }
  return 0;
}

template <class C, int BM, bool LOSS, bool FOLD = false>
int launch_contract_t(TcState* s, int which, double beta, cudaStream_t st) {
  using L = SmemLayout<C::KW, C::TN, C::NF, C::NG, C::NV, C::NS>;
  static_assert(L::kTotal + 1024 <= 232448, "shared memory budget (227 KB)");
  auto kern = tc_contract_kernel<C, BM, LOSS, FOLD>;
  if (!LOSS) s->w_pending = false;       // every update contraction overwrites the partial numerators
  static unsigned long long attr_set_mask = 0;      // per device (one bit each): the attribute is per-device state
  const int smem = L::kTotal + 1024;     // slack so the kernel-visible base can be 1024-aligned
  if (!((attr_set_mask >> (s->device & 63)) & 1ull)) {
    NMF_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_set_mask |= 1ull << (s->device & 63);
  }
  if (C::TN != s->TN || C::RP != s->Rp) { set_error("internal: kernel configuration does not match the plan"); return -1; }
  TcKernelParams p{};
  const Plan& pl = which == 0 ? s->plan_w : s->plan_h;
  p.Mr = (int)(which == 0 ? s->C : s->N);
  p.Nc = (int)(which == 0 ? s->N : s->C);
  p.row_blocks = pl.row_blocks; p.tiles = pl.tiles; p.nchunks = pl.nchunks; p.tiles_per_chunk = pl.tpc;
  p.part = s->part; p.chunk_stride = (int64_t)p.Mr * s->Rp; p.ldp = s->Rp;
  p.part2 = s->part2; p.bm1 = (float)(beta - 1.0); p.bm2 = (float)(beta - 2.0);
  p.exps = s->exps;
  p.ef = which == 0 ? 1 : 2;
  p.eg = which == 0 ? 2 : 1;
  p.loss_part = s->loss_part;
  p.kappa = s->kappa;
  const int items = pl.row_blocks * pl.nchunks;
  const int grid = items < s->num_sms ? items : s->num_sms;
  if (which == 0)
    kern<<<grid, C::kThreads, smem, st>>>(s->tmWf, s->tmHg, s->tmVt, p);
  else
    kern<<<grid, C::kThreads, smem, st>>>(s->tmHf, s->tmWg, s->tmV, p);
  NMF_LAUNCH_CHECK();
  return grid;
}

// Kernel configurations <RP, SPLIT, TN, NF, NG, NV, NS> (224 KB of shared memory each).  Tuning notes in
// profiles/README.md and DESIGN.md 4.1: the V ring must keep >= 3 tiles (>= 64 KB) in flight to cover HBM latency, the G
// ring needs >= 4 stages (a G tile stays resident from its S-MMA to its O-MMA); deeper G rings (5, 6) changed nothing.
using CfgFast64 = Cfg<64, false, 128, 2, 4, 4, 3>;       // F 2x16 | G 4x16 | V 4x32 KB     ; TMEM 3x128 + 64
using CfgSplit64 = Cfg<64, true, 128, 1, 3, 3, 3>;       // F 32 | G 3x32 | V 3x32 KB     ; TMEM 3x128 + 128
using CfgFast128 = Cfg<128, false, 128, 1, 3, 3, 3>;     // F 32 | G 3x32 | V 3x32 KB     ; TMEM 3x128 + 128
using CfgSplit128 = Cfg<128, true, 64, 1, 3, 4, 4>;      // F 64 | G 3x32 | V 4x16 KB     ; TMEM 4x64 + 256
using CfgLoss64 = Cfg<64, false, 128, 2, 4, 4, 2>;       // loss sums, R <= 64 fast: F 2x16 | G 4x16 | V 4x32 KB ; TMEM 2x128
using CfgTwo64 = Cfg<64, false, 128, 2, 3, 4, 2>;        // beta != 1: F 2x16 | G 3x16 | V 4x32 KB ; TMEM 2x128 + 128 + 2x64

// one-output kernels (beta 1: BM = kBmKL, beta 2: BM = kBmEU) over the configuration of this context
template <int BM>
int launch_contract_one(TcState* s, int which, double beta, cudaStream_t st) {
  if (s->Rp == 64) {
    if (!s->split) return launch_contract_t<CfgFast64, BM, false>(s, which, beta, st);
    return launch_contract_t<CfgSplit64, BM, false>(s, which, beta, st);
  }
  if (!s->split) return launch_contract_t<CfgFast128, BM, false>(s, which, beta, st);
  return launch_contract_t<CfgSplit128, BM, false>(s, which, beta, st);
}

// beta 1, W orientation, loss sums folded in (fast, non-split configurations)
int launch_contract_w_fold(TcState* s, cudaStream_t st) {
  if (s->Rp == 64) return launch_contract_t<CfgFast64, kBmKL, false, true>(s, 0, 1.0, st);
  return launch_contract_t<CfgFast128, kBmKL, false, true>(s, 0, 1.0, st);
}

template <int BM>
int launch_loss_bm(TcState* s, double beta, cudaStream_t st) {
  if (s->Rp == 64) {
    if (!s->split) return launch_contract_t<CfgLoss64, BM, true>(s, 1, beta, st);
    return launch_contract_t<CfgSplit64, BM, true>(s, 1, beta, st);
  }
  if (!s->split) return launch_contract_t<CfgFast128, BM, true>(s, 1, beta, st);
  return launch_contract_t<CfgSplit128, BM, true>(s, 1, beta, st);
}

// beta != 1 (and != 2): two-output kernel on the hi halves of the operand copies
int launch_contract_two(TcState* s, int which, double beta, cudaStream_t st) {
  if (!s->part2) NMF_CUDA_CHECK(cudaMalloc(&s->part2, (size_t)s->part_floats * 4));
  int g;
  if (beta == 0.0) g = launch_contract_t<CfgTwo64, kBmIS, false>(s, which, beta, st);
  else if (beta == 0.5) g = launch_contract_t<CfgTwo64, kBm05, false>(s, which, beta, st);
  else if (beta == 1.5) g = launch_contract_t<CfgTwo64, kBm15, false>(s, which, beta, st);
  else g = launch_contract_t<CfgTwo64, kBmGen, false>(s, which, beta, st);
  return g > 0 ? 0 : 2;
}

int launch_contract(TcState* s, int which, double beta, cudaStream_t st) {
  if (beta == 2.0) return launch_contract_one<kBmEU>(s, which, beta, st) > 0 ? 0 : 2;
  if (beta != 1.0) return launch_contract_two(s, which, beta, st);
  return launch_contract_one<kBmKL>(s, which, beta, st) > 0 ? 0 : 2;
}

}  // namespace

int tc_update_w(TcState* s, float* W, const float* H, double beta, double gamma, double l1, double l2,
                cudaStream_t st) {
  // tc_loss_prefetch_w already ran this contraction on these very factors (its numerators are still in `part`)
  const bool reuse = s->w_pending && !s->dirty_w && !s->dirty_h && beta == 1.0;
  s->w_pending = false;
  int rc = ensure_synced(s, W, H, beta, st);
  if (rc) return rc;
  if (!reuse) {
    rc = launch_contract(s, 0, beta, st);
    if (rc) return rc;
  }
  return apply_and_finish(s, 0, W, true, &s->plan_w, beta, gamma, l1, l2, st, nullptr, H);
}

int tc_update_h(TcState* s, const float* W, float* H, double beta, double gamma, double l1, double l2,
                cudaStream_t st) {
  int rc = ensure_synced(s, W, H, beta, st);
  if (rc) return rc;
  rc = launch_contract(s, 1, beta, st);
  if (rc) return rc;
  return apply_and_finish(s, 1, H, true, &s->plan_h, beta, gamma, l1, l2, st, nullptr, W);
}

int tc_iterate(TcState* s, float* W, float* H, double beta, double gamma, double l1, double l2, int n_iter,
               cudaStream_t st) {
  for (int i = 0; i < n_iter; ++i) {
    int rc = tc_update_w(s, W, H, beta, gamma, l1, l2, st);
    if (rc == 0) rc = tc_update_h(s, W, H, beta, gamma, l1, l2, st);
    if (rc) return rc;
  }
  return 0;
}

// Raw update terms of one factor (which = 0: W, 1: H) in one dense buffer: numerator (rows x R; chunk sums, + kappa
// colsum(other) for beta 1, since the kernel accumulated sum (P - kappa) G) followed by colsum(other factor) (R, beta 1) or
// the raw denominator (rows x R).  One contraction launch + one pack launch.
int tc_raw_terms(TcState* s, int which, const float* W, const float* H, double beta, float* out, cudaStream_t st) {
  int rc = ensure_synced(s, W, H, beta, st);
  if (rc) return rc;
  rc = launch_contract(s, which, beta, st);
  if (rc) return rc;
  const int64_t rows = which == 0 ? s->C : s->N;
  const Plan& pl = which == 0 ? s->plan_w : s->plan_h;
  const int64_t RR = rows * s->R;
  const int64_t total = beta == 1.0 ? RR + s->R : 2 * RR;
  w_partial_pack_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, st>>>(
      s->part, beta == 1.0 ? nullptr : s->part2, pl.nchunks, rows * s->Rp, rows, (int)s->R, s->Rp,
      s->colsum + (1 - which) * s->R, s->kappa, out);
  NMF_LAUNCH_CHECK();
  return 0;
}

// Sharded W update, second half: nmf.py:78-92 on the all-reduced buffer with the tensor-core path's own ratio-stage
// kernels, which also rebuild W16 / colsum(W) / exponents (no separate resync pass).
int tc_w_apply(TcState* s, float* W, const float* reduced, double beta, double gamma, double l1, double l2,
               cudaStream_t st) {
  if (!s->has_target) { set_error("tensor-core path: set_target has not been called"); return 3; }
  int rc = apply_and_finish(s, 0, W, true, nullptr, beta, gamma, l1, l2, st, reduced);
  if (rc == 0) s->dirty_w = false;
  return rc;
}

// ---- row-sharded W update over peer memory --------------------------------------------------------------------------------
// contraction -> pack kernel that PUSHES this rank's partial into its slot of every rank's exchange block over NVLink and then
// publishes the iteration counter -> ONE ratio-stage kernel per rank that waits for all counters, sums the slots of its own
// block in rank order and applies nmf.py:78-92 (tc_apply_finish_kernel).  No collective library call and no reduced copy in
// between; slots alternate by iteration parity (a rank can be at most one W update ahead of the slowest: its next push needs
// every rank's counter of the update in between, which that rank publishes after it has read the previous slots).
bool tc_peer_supported(const TcState* s, double beta) {
  return (s->R & 3) == 0 && s->coop_blocks > 0 && tc_supports_partial(s, beta);
}

int tc_peer_alloc(TcState* s, void* handle_out) {
  tc_peer_release(s);
  s->peer_buf_floats = 2 * s->C * s->R;
  const size_t bytes = (64 + 2 * (size_t)kMaxPeers * (size_t)s->peer_buf_floats) * sizeof(float);
  NMF_CUDA_CHECK(cudaMalloc(&s->peer_block, bytes));
  NMF_CUDA_CHECK(cudaMemset(s->peer_block, 0, bytes));
  NMF_CUDA_CHECK(cudaMalloc(&s->peer_err, 2 * sizeof(unsigned int)));      // [0] wait-timeout record, [1] pack-kernel ticket
  NMF_CUDA_CHECK(cudaMemset(s->peer_err, 0, 2 * sizeof(unsigned int)));
  NMF_CUDA_CHECK(cudaDeviceSynchronize());
  cudaIpcMemHandle_t h;
  NMF_CUDA_CHECK(cudaIpcGetMemHandle(&h, s->peer_block));
  static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
  memcpy(handle_out, &h, sizeof(h));
  return 0;
}

int tc_peer_connect(TcState* s, int world, int rank, const void* handles) {
  if (!s->peer_block) { set_error("peer_connect before peer_alloc"); return 3; }
  if (world < 2 || world > kMaxPeers || rank < 0 || rank >= world) { set_error("peer_connect: 2 to 8 ranks"); return 1; }
  unsigned int* flag_ptrs[kMaxPeers] = {};
  for (int p = 0; p < world; ++p) {
    if (p == rank) {
      s->peer_base[p] = s->peer_block;
    } else {
      cudaIpcMemHandle_t h;
      memcpy(&h, static_cast<const char*>(handles) + 64 * p, 64);
      void* ptr = nullptr;
      cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess) {
        s->peer_world = p;             // release what was opened so far
        s->peer_rank = rank;
        tc_peer_release(s);
        set_error(std::string("cudaIpcOpenMemHandle: ") + cudaGetErrorString(e));
        return 2;
      }
      s->peer_base[p] = ptr;
    }
    flag_ptrs[p] = reinterpret_cast<unsigned int*>(s->peer_base[p]);
  }
  s->peer_world = world; s->peer_rank = rank; s->peer_iter = 0;
  NMF_CUDA_CHECK(cudaMalloc(&s->peer_flag_tab, sizeof(flag_ptrs)));
  NMF_CUDA_CHECK(cudaMemcpy(s->peer_flag_tab, flag_ptrs, sizeof(flag_ptrs), cudaMemcpyHostToDevice));
  return 0;
}

int tc_peer_world(const TcState* s) { return s->peer_world; }

int tc_update_w_peer(TcState* s, float* W, const float* H, double beta, double gamma, double l1, double l2,
                     cudaStream_t st) {
  if (s->peer_world < 2) { set_error("peer W update: peers are not connected"); return 3; }
  if (!tc_peer_supported(s, beta)) { set_error("peer W update: unsupported rank / beta"); return 1; }
  int rc = ensure_synced(s, W, H, beta, st);
  if (rc) return rc;
  rc = launch_contract(s, 0, beta, st);
  if (rc) return rc;
  ++s->peer_iter;
  const int64_t slot = 64 + ((int64_t)(s->peer_iter & 1u) * kMaxPeers + s->peer_rank) * s->peer_buf_floats;
  PeerPush push{};
  for (int p = 0; p < s->peer_world; ++p) push.dst[p] = reinterpret_cast<float*>(s->peer_base[p]) + slot;
  const int64_t RR = s->C * s->R;
  const int64_t total = beta == 1.0 ? RR + s->R : 2 * RR;
  w_pack_push_kernel<<<(unsigned)ceil_div(total, 1024), 256, 0, st>>>(
      s->part, beta == 1.0 ? nullptr : s->part2, s->plan_w.nchunks, s->C * s->Rp, s->C, (int)s->R, s->Rp,
      s->colsum + s->R, s->kappa, push, PeerSignal{s->peer_err + 1, s->peer_flag_tab, s->peer_world, s->peer_rank, s->peer_iter});
  NMF_LAUNCH_CHECK();
  const float* mine = reinterpret_cast<const float*>(s->peer_block) + slot;       // layout marker for the ratio stage
  rc = apply_and_finish(s, 0, W, true, nullptr, beta, gamma, l1, l2, st, mine, nullptr, /*peer=*/true);
  if (rc == 0) s->dirty_w = false;
  return rc;
}

// 0: fine; > 0: 1 + the rank whose counter a ratio-stage kernel gave up waiting for (synchronises the stream)
int tc_peer_check(TcState* s, cudaStream_t st) {
  if (!s->peer_err) return 0;
  unsigned int e = 0;
  if (cudaMemcpyAsync(&e, s->peer_err, sizeof(e), cudaMemcpyDeviceToHost, st) != cudaSuccess) return -1;
  if (cudaStreamSynchronize(st) != cudaSuccess) return -1;
  if (e) cudaMemsetAsync(s->peer_err, 0, sizeof(e), st);
  return (int)e;
}

// debugging aid: report (and clear) a recorded mbarrier wait abort; synchronises the stream
int tc_check_wait_abort(cudaStream_t st) {
  if (cudaStreamSynchronize(st) != cudaSuccess) return -1;
  return ptx::check_wait_abort("");
}

int tc_contract_only(TcState* s, const float* W, const float* H, int which, double beta, cudaStream_t st) {
  int rc = ensure_synced(s, W, H, beta, st);
  if (rc) return rc;
  rc = launch_contract(s, which, beta, st);
  if (rc == 0 && s->check_each) {
    if (tc_check_wait_abort(st) > 0) { set_error("mbarrier wait aborted (protocol bug)"); return 2; }
  }
  return rc;
}

bool tc_supports_loss_prefetch(const TcState* s, double beta) {
  return beta == 1.0 && !s->split;
}

// The loss at the current factors from the W update's own contraction (beta 1): one pass over V yields both the loss sums and
// the partial numerators; the next tc_update_w on unchanged factors skips its contraction.
int tc_loss_prefetch_w(TcState* s, const float* W, const float* H, double beta, double* loss_dev, cudaStream_t st) {
  if (!tc_supports_loss_prefetch(s, beta)) return tc_loss(s, W, H, beta, loss_dev, st);
  int rc = ensure_synced(s, W, H, beta, st);
  if (rc) return rc;
  const int grid = launch_contract_w_fold(s, st);
  if (grid <= 0) return 2;
  tc_loss_final_kernel<<<1, 32, 0, st>>>(s->loss_part, grid, s->vconst, s->exps, loss_dev);
  NMF_LAUNCH_CHECK();
  s->w_pending = true;
  return 0;
}

int tc_loss(TcState* s, const float* W, const float* H, double beta, double* loss_dev, cudaStream_t st) {
  int rc = ensure_synced(s, W, H, beta, st);
  if (rc) return rc;
  // S = H W^T over the H-update decomposition (row blocks of H, tiles of W), no second GEMM
  if (beta == 1.0) {
    int grid = launch_loss_bm<kBmKL>(s, beta, st);
    if (grid <= 0) return 2;
    tc_loss_final_kernel<<<1, 32, 0, st>>>(s->loss_part, grid, s->vconst, s->exps, loss_dev);
    NMF_LAUNCH_CHECK();
    return 0;
  }
  if (beta != 2.0 && s->vbeta_for != beta) {      // V-only term of this beta, once per (target, beta)
    v_beta_term_kernel<<<1024, 256, 0, st>>>(s->Vsrc, s->N, s->C, s->ldv, (float)beta, s->vbeta_part);
    NMF_LAUNCH_CHECK();
    sum_blocks_kernel<<<1, 256, 0, st>>>(s->vbeta_part, 1024, s->vbeta);
    NMF_LAUNCH_CHECK();
    s->vbeta_for = beta;
  }
  int grid = beta == 2.0 ? launch_loss_bm<kBmEU>(s, beta, st)
                         : (beta == 0.0 ? launch_loss_bm<kBmIS>(s, beta, st) : launch_loss_bm<kBmGen>(s, beta, st));
  if (grid <= 0) return 2;
  tc_loss_final_beta_kernel<<<1, 32, 0, st>>>(s->loss_part, grid, s->vbeta, beta, (double)s->N * (double)s->C, loss_dev);
  NMF_LAUNCH_CHECK();
  return 0;
}

}  // namespace nmfb200
