// Host-side launchers shared between the translation units (internal; the public ABI is
// include/eims_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/eims_b200.h"
#include "common.cuh"

namespace eims {

// graph.cu
int launch_csr_build(const eims_dataset* ds, const int32_t* ids, int B, int F, int max_nodes, int max_edges,
                     int* gptr, int* eptr, int* gid, int* src, int* dst, int* rowptr, int* col, float* norm,
                     float* x, int* dims, cudaStream_t st, float* a0 = nullptr, int seq = 1,
                     const StepBlock* blk = nullptr,  // non-null: ids and seq are read from the device step block
                     int* bids = nullptr);            // optional: copy of the batch's molecule ids [B]
int launch_layer0_fwd(const int* dims, const float* norm, const float* a0, int F, const float* W, const float* bias,
                      int H, float* z, int max_nodes, cudaStream_t st, const BnFuse* bn = nullptr, float* zero = nullptr,
                      int64_t zero_n4 = 0);
// backward statistics of the BatchNorm whose output gradient the backward-form SpMM writes (see graph.cu)
struct BnBwdFuse {
  const float* z; const float* mean; const float* invstd;  // of that BatchNorm: its input and forward statistics
  double* acc; unsigned int* ticket;                       // bn_partials scratch
  float* dgamma; float* dbeta; float* means;               // outputs: gradients (+=) and the two column means [2][H]
};
int launch_spmm_norm(const int* dims, const int* rowptr, const int* col, const float* norm, const float* h, int H,
                     const float* bn_scale, const float* bn_shift, DropCfg drop, int out_mode, float* out,
                     int max_nodes, cudaStream_t st, const BnBwdFuse* bf = nullptr,
                     const int* gptr = nullptr, int max_graphs = 0, int tile_rows = 0,   // gptr + tile_rows: molecule-tile kernel
                     int64_t lo_off = 0);  // != 0: out = hi plane, out + lo_off = lo plane of a stacked tf32 pair (gemm_tma.cu)
// the molecule-tile kernel itself, whatever the batch size (launch_spmm_norm picks it for large batches only)
int launch_spmm_mol(const int* dims, const int* gptr, const int* rowptr, const int* col, const float* norm, const float* h, int H,
                    const float* bn_scale, const float* bn_shift, DropCfg drop, int out_mode, float* out, int max_graphs,
                    int tile_rows, cudaStream_t st, const BnBwdFuse* bf, int64_t lo_off = 0);
// gradient w.r.t. the atom features: da0 = q0 W0^T ([N, F], q0 from launch_bn_bwd_apply(store_q0)), then dx = D A da0
int launch_layer0_dgrad(const int* dims, const float* q0, int H, const float* W0, int F, float* da0, int max_nodes,
                        cudaStream_t st);
int launch_feat_grad(const int* dims, const int* rowptr, const int* col, const float* norm, const float* da0, int F,
                     float* dx, int max_nodes, cudaStream_t st);
// integrated gradients (eims_attribute_peaks): ig (=|+=) w * D A da0, then ig *= x when x != NULL
int launch_ig_feat_accum(const int* dims, const int* rowptr, const int* col, const float* norm, const float* da0, int F,
                         float w, bool first, const float* x, float* ig, int max_nodes, cudaStream_t st);
// out = alpha * in over the batch's N x F values
int launch_feat_scale(const int* dims, const float* in, int F, float alpha, float* out, int max_nodes, cudaStream_t st);
int launch_readout(const int* dims, const int* gptr, const float* z, int H, const float* bn_scale,
                   const float* bn_shift, int pooling, float* out, int* argmax, int max_graphs, cudaStream_t st,
                   float* zstat = nullptr, const float* bn_mean = nullptr);  // zstat [B][2H]: per graph, column sums of
                                                                             // z - bn_mean and z - bn_mean at the arg-max node (training)

// GEMM problems of the fp32 SIMT kernel (dense.cu) and the tcgen05 kernel (gemm_tc.cu).
// How a GEMM writes C; the values are those of eims_gemm's `accumulate`.
enum GemmAcc : int {
  kGemmStore = 0,             // C = result
  kGemmAdd = 1,               // C += result, atomically (split-K weight gradients)
  kGemmStoreSplit = 2,        // store, but a small grid may split K and add into C, which the launch zeroes first
  kGemmStoreSplitZeroed = 3,  // the same with C already zeroed by the caller
};
// C[M,N] = op(A) op(B) (* row_scale per row, + bias, ReLU); a_mn / b_mn: the operand is stored MN-major.  m_dev / k_dev
// (may be NULL) override M / K with the live sizes on the device.
struct GemmProblem {
  const float* A; int lda, a_mn; const float* B; int ldb, b_mn; float* C; int ldc, M, N, K;
  const int* m_dev; const int* k_dev; const float* row_scale; const float* bias; int relu; GemmAcc accumulate; const BnFuse* bn;
};

// dense.cu
int launch_gemm_simt(const GemmProblem& q, cudaStream_t st);
int64_t bn_scratch_floats(int H, int max_nodes);
int launch_bn_stats(const int* dims, const float* z, int H, const float* gamma, const float* beta, float* rmean,
                    float* rvar, float* mean, float* invstd, float* scale, float* shift, float* partials,
                    int max_nodes, cudaStream_t st);
int launch_bn_eval_coeffs(const float* gamma, const float* beta, const float* rmean, const float* rvar, int H,
                          float* scale, float* shift, cudaStream_t st,
                          float* mean = nullptr, float* invstd = nullptr);  // also: running mean, 1/sqrt(running_var + eps)
// means (the two column means the apply pass subtracts) may be NULL in the statistics passes below: eval mode
int launch_bn_bwd_stats(const int* dims, const float* dh, const float* z, int H, const float* mean, const float* invstd,
                        float* dgamma, float* dbeta, float* means, float* partials, int max_nodes, cudaStream_t st);
// statistics of the TOP layer's BatchNorm backward from per-graph quantities (O(B*H) instead of O(N*H))
int launch_bn_bwd_stats_top(const int* dims, const float* dG, const float* zstat, const int* gptr, int pooling, int H,
                            const float* mean, const float* invstd, float* dgamma, float* dbeta, float* means,
                            float* partials, int max_graphs, cudaStream_t st);
// the zstat [B][2H] that launch_bn_bwd_stats_top reads, for an eval-mode forward (mean: the running mean)
int launch_bn_eval_zstat(const int* dims, const int* gptr, const float* z, int H, const float* mean, const int* argmax,
                         int pooling, float* zstat, int max_graphs, cudaStream_t st);
int launch_bn_bwd_apply(const int* dims, const float* dh, const float* dG, const int* gid, const int* gptr,
                        const int* argmax, int pooling, const float* z, int H, const float* mean, const float* invstd,
                        const float* gamma, const float* norm, float* dbias, const float* means, float* q, int max_nodes,
                        cudaStream_t st, const float* a0 = nullptr, int F = 0, float* dW0 = nullptr,
                        int64_t q_lo_off = 0,     // != 0: q as stacked tf32 hi / lo planes
                        bool store_q0 = false);   // layer 0 (dW0 set): also store q_0 into q as plain fp32
// the data-only eval backward (eims_attribute_peaks): q only, no bias gradient / dW0 / column means
int launch_bn_dgrad_apply(const int* dims, const float* dh, const float* dG, const int* gid, const int* gptr,
                          const int* argmax, int pooling, const float* z, int H, const float* mean, const float* invstd,
                          const float* gamma, const float* norm, float* q, int max_nodes, cudaStream_t st,
                          int64_t q_lo_off = 0);
int launch_ln_fwd(const int* dims, const float* u, int W, const float* gamma, const float* beta, DropCfg drop, float* y,
                  float* stats, int max_graphs, cudaStream_t st);
int launch_ln_bwd(const int* dims, const float* u, const float* y, const float* dy, int W, const float* gamma,
                  const float* stats, float drop_scale, float* du, float* dgamma, float* dbeta, float* dbias,
                  int max_graphs, cudaStream_t st);
// eval mode, data gradient only (no dgamma / dbeta / bias gradient, no dropout)
int launch_ln_dgrad(const int* dims, const float* u, const float* y, const float* dy, int W, const float* gamma,
                    const float* stats, float* du, int max_graphs, cudaStream_t st);
// peaks of eims_attribute_peaks: dy2[r] = p(1-p) W3[bins[r]]; bins / prob from the top-k table (entry r mod k);
// prob[r] = sigmoid(logits[r, bins[r]])
int launch_peak_head_dgrad(const int* dims, const float* logits, int M, const int* bins, const float* W3, int H, float* dy2,
                           int max_graphs, cudaStream_t st);
int launch_peak_select(const int* dims, const int* idx, const float* val, int k, int* bins, float* prob, int max_graphs,
                       cudaStream_t st);
int launch_peak_prob(const int* dims, const float* logits, int M, const int* bins, float* prob, int max_graphs,
                     cudaStream_t st);
int launch_loss(const int* dims, const float* logits, const float* targets, const int* target_rows, int M,
                int loss_kind, float* prob, float* dlogits, float* row_loss, float* row_cos, int max_graphs,
                cudaStream_t st, float* metrics = nullptr, unsigned int* ticket = nullptr,
                const eims_peaks* peaks = nullptr);
int launch_peaks_to_spectrum(const eims_peaks* pk, const int* rows, int num_rows, int M, float* out, cudaStream_t st);
int launch_topk_peaks(const float* spectra, int num_rows, int M, int k, int* idx_out, float* val_out, cudaStream_t st);
int launch_sigmoid(const int* dims, const float* logits, int M, float* prob, int max_graphs, cudaStream_t st);
int launch_dprob_to_dlogits(const int* dims, const float* prob, const float* dprob, int M, float* dlogits,
                            int max_graphs, cudaStream_t st);
int launch_metrics(const int* dims, const float* row_loss, const float* row_cos, int M, float* metrics, cudaStream_t st);
int launch_colsum(const int* dims, int dim_slot, const float* in, int C, int ld, float* out, int max_rows, cudaStream_t st);
int launch_adamw(float* p, float* g, float* m, float* v, int64_t n, const eims_step* s, cudaStream_t st,
                 const StepBlock* blk = nullptr);  // blk: the scalars are read from the device step block
int launch_step_blocks_store(const StepBlockPack& v, StepBlock* dst, int n, cudaStream_t st);
int launch_dropout_mask(DropCfg d, int rows, int W, float* out, cudaStream_t st);

// gemm_tc.cu  (tcgen05 / TMEM, 3xTF32)
int launch_gemm_tc(const GemmProblem& q, cudaStream_t st);
int launch_gemm_tc_pair(const GemmProblem& p0, const GemmProblem& p1, cudaStream_t st);

// gemm_tma.cu  (tcgen05 / TMEM, 3xTF32 on pre-split hi / lo operand planes fed by the tensor-map copy engine, persistent)
struct alignas(64) TmaMap { uint8_t bytes[128]; };  // a CUtensorMap (driver type) kept opaque outside gemm_tma.cu
// map over the stacked planes [2][rows][ld] (plane_stride floats apart) of a row-major operand with `cols` columns:
// mn_major = 0 -> the rows are the operand's M / N index (box_rows of them per tile), 1 -> the rows are its K index
int tma_make_map(TmaMap* out, const float* planes, int64_t plane_stride, int rows, int cols, int ld, int box_rows, int mn_major);
bool gemm_tma_enabled();  // the driver offers cuTensorMapEncodeTiled
constexpr int kTmaBRows = 128;  // box rows of a K-major B map: each CTA of a pair stages half of a 256-column tile
struct GemmTmaProblem {
  const TmaMap* ta; const TmaMap* tb; float* C; int ldc, a_mn, b_mn, M, N, K;
  const int* m_dev; const int* k_dev; const float* row_scale; const float* bias; int relu, red; const BnFuse* bn;
};
bool gemm_tma_supports(const GemmTmaProblem& q);
// one launch: a store problem (red = 0) and / or a split-K problem (red = 1: partial sums added into C)
int launch_gemm_tma(const GemmTmaProblem* p0, const GemmTmaProblem* p1, cudaStream_t st);
int launch_split_planes(const float* src, float* hi, float* lo, int64_t n, cudaStream_t st, bool chained);

}  // namespace eims
