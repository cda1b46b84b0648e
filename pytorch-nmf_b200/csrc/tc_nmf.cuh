// Tensor-core (tcgen05 / TMEM / TMA) path of the dense NMF update -- interface used by capi.cu.
#pragma once
#include "common.cuh"

namespace nmfb200 {

struct TcState;

// shapes the tcgen05 kernels accept (rank padded to 64 or 128 columns)
bool tc_shape_supported(int64_t N, int64_t C, int64_t R);
int tc_create(TcState** out, int device, int64_t N, int64_t C, int64_t R, bool split);
void tc_destroy(TcState* s);
bool tc_supports_beta(const TcState* s, double beta);
// row-sharded partials: beta 2 keeps the fp32 contraction (its numerator needs the Gram matrix of the global H)
bool tc_supports_partial(const TcState* s, double beta);
// minmax_dev: device float[2] = {min(V), max(V)} already queued on `st`
int tc_set_target(TcState* s, const float* V, int64_t ldv, const float* minmax_dev, cudaStream_t st);
// number of positive target entries that the scaled fp16 copy holds only as subnormals / zero (synchronises `st`)
int tc_target_lossy(TcState* s, unsigned long long* count, cudaStream_t st);
// sum of the registered target (synchronises `st`)
int tc_target_sum(TcState* s, double* vsum, cudaStream_t st);
// the fp32 factor changed outside the tensor-core path: operand copies must be rebuilt before use
void tc_mark_dirty(TcState* s, bool w, bool h);
int tc_update_w(TcState* s, float* W, const float* H, double beta, double gamma, double l1, double l2,
                cudaStream_t st);
int tc_update_h(TcState* s, const float* W, float* H, double beta, double gamma, double l1, double l2,
                cudaStream_t st);
int tc_iterate(TcState* s, float* W, float* H, double beta, double gamma, double l1, double l2, int n_iter,
               cudaStream_t st);
// raw update terms of one factor (which = 0: W, 1: H; which = 0 is the row-sharded W update's partial):
// [numerator rows x R | colsum(other) R (beta 1) or denominator rows x R]
int tc_raw_terms(TcState* s, int which, const float* W, const float* H, double beta, float* out, cudaStream_t st);
int tc_w_apply(TcState* s, float* W, const float* reduced, double beta, double gamma, double l1, double l2,
               cudaStream_t st);
// row-sharded W update over peer memory (one NVLink domain, 2 to 8 ranks): allocate this rank's exchange block and export its
// 64-byte CUDA IPC handle; open the other ranks' blocks (`handles`: world x 64 bytes, in rank order); then every rank calls
// tc_update_w_peer for every W update (collective).  tc_peer_check: > 0 if a kernel gave up waiting for a rank.
bool tc_peer_supported(const TcState* s, double beta);
int tc_peer_alloc(TcState* s, void* handle_out);
int tc_peer_connect(TcState* s, int world, int rank, const void* handles);
int tc_peer_world(const TcState* s);
void tc_peer_release(TcState* s);
int tc_update_w_peer(TcState* s, float* W, const float* H, double beta, double gamma, double l1, double l2,
                     cudaStream_t st);
int tc_peer_check(TcState* s, cudaStream_t st);
int tc_contract_only(TcState* s, const float* W, const float* H, int which, double beta, cudaStream_t st);
// debugging / health: report (and clear) a recorded mbarrier wait abort; synchronises the stream
int tc_check_wait_abort(cudaStream_t st);
int tc_loss(TcState* s, const float* W, const float* H, double beta, double* loss_dev, cudaStream_t st);
// the same value out of the W update's own contraction pass (beta 1, non-split); the next tc_update_w on unchanged factors
// reuses the partial numerators.  Falls back to tc_loss where the fold is not built.
int tc_loss_prefetch_w(TcState* s, const float* W, const float* H, double beta, double* loss_dev, cudaStream_t st);

}  // namespace nmfb200
