// NMFD on tcgen05 tensor cores (beta = 1): im2col-free sliding GEMMs for kernels of up to 128 shifts -- interface used by
// capi.cu.  See tc_nmfd.cu.
#pragma once
#include "common.cuh"

namespace nmfb200 {

struct TcNmfdState;

// shapes the kernels compute: one sliding axis, T <= 128 (every shift of wgrad in one accumulator), R <= 256
bool tc_nmfd_shape_supported(const NmfdShape& d);
int tc_nmfd_create(TcNmfdState** out, const NmfdShape& d);
void tc_nmfd_destroy(TcNmfdState* s);
// sum(V) for the centring constant kappa (also returned to the host: synchronises `st`)
int tc_nmfd_set_target(TcNmfdState* s, const float* V, double* vsum_host, cudaStream_t st);
// brings the fp16 operand copies / column sums / kappa up to date with whichever factor changed since the last call, then
// either writes the centred ratio tile (V / (WH + eps) - kappa) 2^p for the following wgrad / dgrad, or (loss) reduces
// metrics.kl_div
int tc_nmfd_recon(TcNmfdState* s, const float* V, const float* W, const float* H, bool loss, double* loss_dev,
                  cudaStream_t st);
// split-K partial numerators from the ratio tile of the last recon: W side [nsplit][C][R][T], H side [nsplit][B][R][Lin]
// (without the kappa * colsum term, which the ratio stage adds: ApplyArgs::kappa / kappa_vec)
int tc_nmfd_wgrad(TcNmfdState* s, const float** part, int* nsplit, cudaStream_t st);
int tc_nmfd_dgrad(TcNmfdState* s, const float** part, int* nsplit, cudaStream_t st);
// [colsum_W (R) | colsum_H (R)] of the factors as of the last recon (the KL denominators, nmf.py:122-131)
const float* tc_nmfd_colsum(const TcNmfdState* s);
// the ratio stage is about to rewrite W (which = 0) or H (1): slot to atomicMax the new values into (ApplyArgs::absmax_bits)
unsigned int* tc_nmfd_begin_update(TcNmfdState* s, int which, cudaStream_t st);
// the factors were changed outside the library: refresh everything at the next recon
void tc_nmfd_mark_dirty(TcNmfdState* s);
const float* tc_nmfd_kappa(const TcNmfdState* s);
// after a stream synchronise: 1 if an NMFD kernel aborted an internal barrier wait since the last check (record cleared)
int tc_nmfd_check_wait_abort();

}  // namespace nmfb200
