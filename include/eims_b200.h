/*
 * eims_b200.h - C ABI of the B200-native GCN EI-MS hot path.
 *
 * The reference (turnDeep/Computational-Chemistry-AI, templates/ms-pred-gcn-eims-cupy.py,
 * "GCN:n" below) has no FFI: the path is ordinary Python calls into DGL / torch / CuPy.
 * Each entry point here names the reference call(s) it replaces.  The Python host layer
 * (computational-chemistry-ai_b200/eims_b200) binds these with ctypes and mirrors the
 * script's own interface (Config, collate_fn, GCNSpectrum, train_model, predict_spectrum).
 *
 * Conventions
 *   - plain pointers and sizes only; every device pointer is caller-owned (torch allocates);
 *   - every function returns 0 on success, <0 on error (never throws); eims_last_error()
 *     gives the message for the calling thread;
 *   - all work is enqueued on the given cudaStream_t and is asynchronous; the library
 *     allocates no device memory (the workspace size comes from eims_plan_workspace_bytes);
 *   - a plan may be used from one thread at a time;
 *   - built for sm_100a only: there is no CPU path and no other GPU path.
 */
#ifndef EIMS_B200_H_
#define EIMS_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* eims_stream_t; /* == cudaStream_t */
typedef struct eims_plan eims_plan;

enum {
  EIMS_OK = 0,
  EIMS_ERR_ARG = -1,       /* bad argument / unsupported dimension */
  EIMS_ERR_CUDA = -2,      /* a CUDA runtime call failed */
  EIMS_ERR_CAPACITY = -3,  /* batch exceeds the plan's max_graphs / max_nodes / max_edges */
  EIMS_ERR_ZERO_DEGREE = -4, /* an atom without bonds: DGL GraphConv raises (GCN:316,359) */
  EIMS_ERR_STATE = -5      /* call order (e.g. backward before forward, plan not bound) */
};

enum { EIMS_POOL_SUM = 0, EIMS_POOL_MEAN = 1, EIMS_POOL_MAX = 2, EIMS_POOL_COMBINED = 3 };
enum { EIMS_LOSS_MSE = 0 /* GCN:393 */, EIMS_LOSS_COSINE = 1 /* north-star variant */ };
enum { EIMS_BWD_ALL = 0, EIMS_BWD_HEAD = 1 /* spectrum_predictor + readout */, EIMS_BWD_GCN = 2 /* GCN layers */ };
enum { EIMS_GEMM_TCGEN05 = 0 /* 3xTF32 tensor-core path */, EIMS_GEMM_FP32_SIMT = 1 /* CUDA-core check path */ };

/* Model hyper-parameters: `Config` GCN:73-101 + node_feat_dim (GCN:580,603). */
typedef struct {
  int32_t node_feat_dim;  /* 6 */
  int32_t hidden_dim;     /* multiple of 64 */
  int32_t num_gcn_layers; /* >= 1 */
  int32_t max_mz;         /* multiple of 4 */
  int32_t pooling;        /* EIMS_POOL_* (GCN:325-338) */
  float dropout;          /* GCN:88 */
} eims_dims;

/* A packed set of molecules in device memory (a whole data set, or one uploaded batch).
 * Molecule g owns atoms [node_ptr[g], node_ptr[g+1]) and bonds [bond_ptr[g], bond_ptr[g+1]);
 * bond ends are molecule-local atom indices in RDKit bond order (GCN:139-143).
 * `targets` is the dense [num_mols, max_mz] spectrum matrix of GCN:256 (may be NULL for
 * inference). */
typedef struct {
  const int64_t* node_ptr;
  const int64_t* bond_ptr;
  const float* feat; /* [total atoms, node_feat_dim], get_atom_features order GCN:113-122 */
  const int32_t* bond_begin;
  const int32_t* bond_end;
  const float* targets;
  int64_t num_mols;
  const struct eims_peaks* peaks; /* optional: the target spectra as peak lists; used when targets == NULL */
} eims_dataset;

/* Peak lists of a set of spectra - what OptimizedEIMSDataset.load_peaks (GCN:260-278) returns per
 * molecule - stored flat: spectrum s owns peaks [peak_ptr[s], peak_ptr[s+1]).  m/z values are
 * float32 (what the reference's CuPy branch rounds, GCN:176-179) or float64 (what its NumPy
 * branch rounds, GCN:193-196); intensities are float32 in both (GCN:171,191). */
typedef struct eims_peaks {
  const int64_t* peak_ptr;
  const void* mz;
  const float* intensity;
  int32_t mz_is_f64;
  int64_t num_spectra;
} eims_peaks;

/* Per-step optimiser scalars, computed on the host exactly as torch's AdamW + OneCycleLR
 * do (GCN:385-391, 429-431): lr and beta1 follow the one-cycle schedule. */
typedef struct {
  float lr, beta1, beta2, eps, weight_decay;
  float grad_scale;  /* 1/world_size for data-parallel training, else 1 */
  int32_t step;      /* 1-based optimiser step count t */
  uint64_t seed;     /* dropout stream seed; the mask is a function of (seed, step, site, element) */
} eims_step;

/* ---------------------------------------------------------------- misc */
int eims_version(void);
const char* eims_last_error(void);
int eims_device_check(void); /* 0 iff the current device is sm_100 */

/* Flat parameter buffer: the 4L+10 trainable tensors in `model.parameters()` order
 * (= state_dict order without BN buffers, SURVEY A.6).  offsets has n_tensors+1 entries. */
int64_t eims_param_count(const eims_dims* d);
int eims_param_num_tensors(const eims_dims* d);
int eims_param_layout(const eims_dims* d, int64_t* offsets, int32_t n_entries);

/* ---------------------------------------------------------------- stand-alone kernels
 * (each is also a stage of eims_train_step; exposed for per-kernel parity tests) */

/* CuPySpectrumProcessor.peaks_to_spectrum_batch (GCN:166-205) on the device: for output row b
 * the spectrum rows[b] (b itself when rows == NULL) of `pk` is binned - bin = round-half-even(m/z),
 * bins outside [0, max_mz) dropped, duplicates max-merged (intensities <= 0 and NaN leave the
 * zero-initialised bin as it is, like the reference's max()), row divided by its maximum
 * (by 1 when the row is all zero).  Bit-exact with the reference's loops.  out is [num_rows, max_mz]. */
int eims_peaks_to_spectrum(const eims_peaks* pk, const int32_t* rows, int32_t num_rows, int32_t max_mz,
                           float* out, eims_stream_t stream);

/* The peak report of `--mode predict` (GCN:610-613: np.argmax and np.argsort(spectrum)[-5:][::-1])
 * for a batch of predicted spectra [num_rows, max_mz]: the k largest bins of every row, value
 * descending; exact ties go to the higher bin (= a stable argsort; the reference's default-kind
 * argsort leaves tie order unspecified).  idx_out [num_rows, k] int32; val_out [num_rows, k] or NULL. */
int eims_topk_peaks(const float* spectra, int32_t num_rows, int32_t max_mz, int32_t k,
                    int32_t* idx_out, float* val_out, eims_stream_t stream);


/* K1  replaces collate_fn -> dgl.batch (GCN:292-297), the in-degree pass and the
 * degree normalisation of DGL GraphConv.  Outputs (all int32 / fp32, device):
 *   gptr[B+1] node offset per graph, eptr[B+1] edge offset per graph, gid[N],
 *   src[E], dst[E] (reference edge order), rowptr[N+1], col[E] (CSR by destination,
 *   ascending edge id inside a row), norm[N] = fl(1/fl(sqrt(max(deg,1)))), x[N,F],
 *   dims[8] = {B, N, E, zero_degree_flag, overflow_flag, 0,0,0}. */
int eims_csr_build(const eims_dataset* ds, const int32_t* mol_ids, int32_t num_graphs,
                   int32_t node_feat_dim, int32_t max_nodes, int32_t max_edges,
                   int32_t* gptr, int32_t* eptr, int32_t* gid, int32_t* src, int32_t* dst,
                   int32_t* rowptr, int32_t* col, float* norm, float* x, int32_t* dims,
                   eims_stream_t stream);

/* K2  replaces DGL update_all(copy_u, sum) with the source-side normalisation
 * (GraphConv, GCN:359):  out[i,:] = sum_{j in row i} fl(f(h[j,:]) * norm[j])  where
 * f(x) = x*scale+shift (BatchNorm apply, may be NULL) followed by the dropout mask of
 * `site` (skipped when drop_p == 0).  With out_scale_norm != 0 (the backward form,
 * dh = (A da) * c) the gathered rows are summed unscaled and the result row is scaled by
 * norm[i] and by the dropout mask of row i. */
int eims_spmm_norm(const int32_t* dims, const int32_t* rowptr, const int32_t* col, const float* norm,
                   const float* h, int32_t width, const float* bn_scale, const float* bn_shift,
                   float drop_p, uint64_t seed, int32_t step, int32_t site,
                   int32_t out_scale_norm, float* out, int32_t max_nodes, eims_stream_t stream);

/* K2, molecule tiles: the same result bit for bit, computed block-per-molecule with the molecule's [n_g, width] tile
 * of h staged in shared memory by the bulk async-copy engine (each row read once instead of once per neighbour; the
 * BatchNorm / dropout / degree-norm transform applied once per element).  gptr[B+1] = node offset per graph (K1);
 * tile_rows = rows of the shared tile (<= 128; molecules with more atoms take the gather path in the same kernel);
 * width must be a multiple of 128.  This is what the plan's forward / backward use. */
int eims_spmm_norm_mol(const int32_t* dims, const int32_t* gptr, const int32_t* rowptr, const int32_t* col, const float* norm,
                       const float* h, int32_t width, const float* bn_scale, const float* bn_shift, float drop_p, uint64_t seed,
                       int32_t step, int32_t site, int32_t out_scale_norm, float* out, int32_t max_nodes, int32_t max_graphs,
                       int32_t tile_rows, eims_stream_t stream);

/* K3/K6  C[M,N] = op(A)[M,K] * op(B)[K,N] in fp32-grade arithmetic.
 * a_mn_major: 0 -> A stored [M,K] row-major (lda), 1 -> stored [K,M] row-major (lda).
 * b_mn_major: 0 -> B stored [N,K] row-major (ldb) (nn.Linear weight), 1 -> stored [K,N]
 * row-major (GraphConv weight).  Epilogue: C = act(acc * row_scale[m] + bias[n]);
 * row_scale / bias may be NULL; relu != 0 applies max(.,0); accumulate = 1 adds into C
 * atomically (split-K weight gradients), accumulate = 2 stores but lets a small grid split K
 * (C is zeroed first; summation order then varies run to run), accumulate = 3 the same with C already zeroed by the caller.  m_dev / k_dev (may be NULL) override M / K with
 * a device-side int (the number of atoms of the current batch).
 * backend: EIMS_GEMM_TCGEN05 or EIMS_GEMM_FP32_SIMT. */
int eims_gemm(int32_t backend, const float* A, int32_t lda, int32_t a_mn_major,
              const float* B, int32_t ldb, int32_t b_mn_major, float* C, int32_t ldc,
              int32_t M, int32_t N, int32_t K, const int32_t* m_dev, const int32_t* k_dev,
              const float* row_scale, const float* bias, int32_t relu, int32_t accumulate,
              eims_stream_t stream);

/* K3/K6 on pre-split operand planes (csrc/gemm_tma.cu): the same products as eims_gemm, computed by the persistent
 * kernel that the plan uses for the GraphConv layers (GCN:316,359 forward, and their weight / data gradients): every
 * operand is first split into stacked tf32 hi / lo planes (inside `scratch`; in the plan the kernels that produce the
 * operands write the planes directly), the planes travel global -> shared by cp.async.bulk.tensor, and one CTA per SM
 * walks over the output tiles of a store problem (accumulate = 0) and / or the k-slices of a split-K problem
 * (accumulate = 1, partial sums added into C), dealt out on the device from the live sizes.  p1 may be NULL; with two
 * problems exactly one must have accumulate = 1.  Needs N % 256 == 0, ldc % 4 == 0, K <= 2048 for the store problem (K > 512
 * keeps the correction products in a second accumulator and gives up the overlap of epilogue and main loop), lda /
 * ldb % 4 == 0; for a split-K problem with a live k_dev < K the operand rows in [k_dev, K) must be finite. */
typedef struct {
  const float* A; int32_t lda, a_mn_major;
  const float* B; int32_t ldb, b_mn_major;
  float* C; int32_t ldc;
  int32_t M, N, K;
  const int32_t* m_dev; const int32_t* k_dev;
  const float* row_scale; const float* bias;
  int32_t relu, accumulate;
} eims_gemm_problem;
int64_t eims_gemm_planes_scratch_bytes(const eims_gemm_problem* p0, const eims_gemm_problem* p1);
int eims_gemm_planes(const eims_gemm_problem* p0, const eims_gemm_problem* p1, void* scratch, int64_t scratch_bytes,
                     eims_stream_t stream);

/* BatchNorm1d training statistics over the N atoms of the batch (GCN:361):
 * mean / biased var per column -> scale = gamma*invstd, shift = beta - mean*scale,
 * saved mean & invstd, running stats update (momentum 0.1, unbiased var).  `partials`
 * is scratch of eims_bn_scratch_floats(width, max_nodes) floats. */
int64_t eims_bn_scratch_floats(int32_t width, int32_t max_nodes);
int eims_bn_stats(const int32_t* dims, const float* z, int32_t width, const float* gamma, const float* beta,
                  float* running_mean, float* running_var, float* mean, float* invstd,
                  float* scale, float* shift, float* partials, int32_t max_nodes, eims_stream_t stream);

/* K5  replaces SumPooling / AvgPooling / MaxPooling (+ torch.cat) GCN:366-371 with the
 * last layer's BatchNorm apply fused in.  out[B, pool_dim]; argmax[B,H] = first maximum. */
int eims_readout(const int32_t* dims, const int32_t* gptr, const float* z, int32_t width,
                 const float* bn_scale, const float* bn_shift, int32_t pooling,
                 float* out, int32_t* argmax, int32_t max_graphs, eims_stream_t stream);

/* K7  replaces Sigmoid (GCN:351) + nn.MSELoss (GCN:393,427) + cosine_similarity_batch
 * (GCN:213-215) and their gradient.  logits[B,M] -> prob[B,M]; target row of graph b is
 * targets[target_rows ? target_rows[b] : b].  row_loss[b] = sum_m (p-t)^2, row_cos[b];
 * dlogits (may be NULL) = dLoss/dlogits for loss_kind, mean over the batch. */
int eims_loss_mse_cos(const int32_t* dims, const float* logits, const float* targets,
                      const int32_t* target_rows, int32_t max_mz, int32_t loss_kind,
                      float* prob, float* dlogits, float* row_loss, float* row_cos,
                      int32_t max_graphs, eims_stream_t stream);

/* K8  replaces optimizer.zero_grad + AdamW.step (GCN:414,429) over the flat buffers.
 * g is scaled by s->grad_scale first and zeroed afterwards. */
int eims_adamw_flat(float* p, float* g, float* m, float* v, int64_t n, const eims_step* s,
                    eims_stream_t stream);

/* Materialise the dropout keep-mask (0/1 floats) of a site, for tests. */
int eims_dropout_mask(float drop_p, uint64_t seed, int32_t step, int32_t site,
                      int32_t rows, int32_t width, float* out, eims_stream_t stream);

/* ---------------------------------------------------------------- host-side collate
 * For callers whose data set lives in HOST memory (the reference's case): replaces collate_fn -> dgl.batch +
 * torch.stack (GCN:292-297) and the DataLoader's pin_memory copy (GCN:567).  `ds` holds HOST pointers here; the
 * batch `ids` (NULL = 0..n-1) is gathered into the caller's (pinned) buffer `out` in the packed layout that
 * eims_batch_build reads after ONE host-to-device copy of `lay->nbytes` bytes; section offsets (bytes, 256-aligned,
 * -1 = absent) come back in `lay`.  Targets: dense rows when ds->targets != NULL, else the peak lists of ds->peaks.
 * Returns EIMS_ERR_CAPACITY (with lay->nbytes = the size needed) when `out` is too small.  Pure host code. */
typedef struct {
  int64_t node_ptr, bond_ptr, bond_begin, bond_end, feat, targets, peak_ptr, peak_mz, peak_inten, nbytes;
  int32_t num_graphs, num_nodes, num_edges, feat_dim, mz_is_f64;
} eims_host_batch;
int eims_host_pack_batch(const eims_dataset* ds, const int32_t* ids, int32_t n, int32_t node_feat_dim, int32_t max_mz,
                         void* out, int64_t capacity, eims_host_batch* lay);
/* The same with a FIXED layout: sections sized for cap_nodes atoms / cap_bonds bonds / cap_peaks peaks, so every batch
 * of n molecules has the same section offsets and nbytes - constant device pointers after the upload, which is what a
 * captured CUDA graph (copy + K1 + step, replayed) needs.  EIMS_ERR_CAPACITY when the batch does not fit; `lay` then
 * still holds the fixed layout and the batch's true num_nodes / num_edges, so a layout query may name any molecules. */
int eims_host_pack_batch_fixed(const eims_dataset* ds, const int32_t* ids, int32_t n, int32_t node_feat_dim, int32_t max_mz,
                               int64_t cap_nodes, int64_t cap_bonds, int64_t cap_peaks, void* out, int64_t capacity,
                               eims_host_batch* lay);

/* ---------------------------------------------------------------- plan: the whole path */
int eims_plan_create(const eims_dims* d, int32_t max_graphs, int32_t max_nodes, int32_t max_edges,
                     eims_plan** out);
int eims_plan_destroy(eims_plan* p);
int64_t eims_plan_workspace_bytes(const eims_plan* p);
int eims_plan_bind(eims_plan* p, void* workspace, int64_t bytes);
int eims_plan_set_gemm_backend(eims_plan* p, int32_t backend);
/* Which kernel runs the GraphConv products (GCN:316,359 and their gradients) on the tensor-core backend:
 * EIMS_PLANES_AUTO (default) - the persistent planes kernel (csrc/gemm_tma.cu: operands pre-split into tf32 hi / lo
 * planes by their producers, fed by cp.async.bulk.tensor, CTA pairs) for plans sized for large batches (>= 4 output
 * tiles per SM), the in-kernel-split kernel (csrc/gemm_tc.cu) otherwise; EIMS_PLANES_OFF / EIMS_PLANES_ON force one.
 * EIMS_ERR_STATE if the planes path is asked for but the plan's shapes do not allow it (hidden_dim % 256 != 0). */
#define EIMS_PLANES_AUTO (-1)
#define EIMS_PLANES_OFF 0
#define EIMS_PLANES_ON 1
int eims_plan_set_gemm_planes(eims_plan* p, int32_t mode);

/* Named views into the bound workspace (tests / host layer).  EIMS_ERR_STATE before eims_plan_bind,
 * EIMS_ERR_ARG for an unknown name.  Names:
 *   batch tables, held twice: "dims","gptr","eptr","gid","bids","src","dst","rowptr","col","norm","x","a0"
 *     - the bare name is the set the calls enqueued next use, "<name>#0" / "<name>#1" a given set;
 *   per GCN layer l: "a<l>" (l >= 1),"z<l>","bn_mean<l>","bn_invstd<l>","bn_scale<l>","bn_shift<l>";
 *   "flags","argmax","bn_means2","bn_partials","readout","zstat","u1","u2","logits","dy2","dy1","dG",
 *   "y1","ln1","y2","ln2","prob","dlogits","row_loss","row_cos","dh","q","da";
 *   "wplanes" (plans whose shapes allow the planes GEMM only). */
int eims_plan_buffer(eims_plan* p, const char* name, void** ptr, int64_t* bytes);

/* K1 on the plan's buffers. */
int eims_batch_build(eims_plan* p, const eims_dataset* ds, const int32_t* mol_ids,
                     int32_t num_graphs, eims_stream_t stream);

/* GCNSpectrum.forward (GCN:354-376) on the batch built last.  training != 0: batch
 * statistics + dropout + everything backward needs is kept; bn_running [L][2][H]
 * (running_mean, running_var) is updated.  Result: "logits" and (after eims_loss or
 * eims_sigmoid) "prob". */
int eims_forward(eims_plan* p, const float* params, float* bn_running, int32_t training,
                 const eims_step* s, eims_stream_t stream);
int eims_sigmoid(eims_plan* p, eims_stream_t stream); /* prob = sigmoid(logits), inference */
/* Targets as peak lists: after this call eims_loss / eims_train_step_built accept targets == NULL
 * and bin row target_rows[b] of `pk` on the fly inside the loss kernel (same arithmetic as
 * eims_peaks_to_spectrum), so a training set keeps ~1 KB of peaks per molecule in HBM instead
 * of a 4*max_mz-byte dense row.  pk == NULL switches back.  The struct is copied; the arrays
 * it points to must stay alive. */
int eims_plan_set_peak_targets(eims_plan* p, const eims_peaks* pk);
int eims_loss(eims_plan* p, const float* targets, const int32_t* target_rows, int32_t loss_kind,
              int32_t want_grad, eims_stream_t stream);
/* dprob: optional [B,M] gradient w.r.t. the spectrum (autograd use); NULL = use the
 * dlogits left by eims_loss(want_grad=1).  Gradients are ADDED into grads (flat, zeroed by
 * eims_adamw_flat / the caller).  Training-mode forwards only (EIMS_ERR_STATE after an eval
 * forward); eims_backward_feat also differentiates eval-mode forwards and the atom features. */
int eims_backward(eims_plan* p, const float* params, const float* dprob, float* grads,
                  eims_stream_t stream);
/* The backward of the forward enqueued last, training OR eval mode, optionally down to the atom features.
 * dprob [B,M]: gradient w.r.t. the spectrum.  It may be NULL only after eims_loss(want_grad=1) in training mode.
 * Parameter gradients are ADDED into grads, as in eims_backward.  In eval mode BatchNorm is the affine map
 * of the running statistics, dropout is off, and running statistics are not touched.
 * dfeat (may be NULL): d/dx of the batch's atom features, [N, F] in batch order, rows [0, N) overwritten. */
int eims_backward_feat(eims_plan* p, const float* params, const float* dprob, float* grads, float* dfeat,
                       eims_stream_t stream);
/* Per-atom attribution of each graph's top predicted peak by integrated gradients (IG), on the batch built last.
 * Definition (new functionality; the reference has no attribution):
 *   - eval mode: BatchNorm uses the running statistics, dropout is off;
 *   - baseline: all-zero atom features on the same graph;
 *   - the peak bin m_r of graph r is the (r mod k)-th largest bin of graph r's own predicted spectrum (the report of
 *     eims_topk_peaks: value descending, exact ties to the higher bin);
 *   - midpoint rule with S = steps points, alpha_s = (s + 1/2) / S, weight 1/S:
 *       ig[i, f] = x[i, f] * (1/S) * sum_s  d prob_{m_r} / d x[i, f]  at alpha_s * X      (i an atom of graph r)
 *     so that sum over graph r's atoms and features of ig ~= peak_prob[r] - base_prob[r] (completeness).
 * A caller that puts each molecule k times in a row (replica j of molecule g is graph g*k + j) gets all k peaks of every
 * molecule from one call.  Outputs: bins[B] (m_r), peak_prob[B] (prob_{m_r}(X)), base_prob[B] (prob_{m_r}(0)), ig[N, F]
 * in batch order; rows past the batch are not written.
 * scratch: caller-owned device memory, 256-byte aligned, of at least 4*N*F + 8*B*k + 512 bytes with N = max_nodes and
 * B = max_graphs of the plan (an unscaled copy of K1's aggregate a0 and the top-k table).
 * Each path point is an eval forward plus a backward to the atom features that computes no parameter gradient.  No
 * float atomics: a molecule's outputs do not depend on the other graphs of the batch.
 * EIMS_ERR_ARG: a NULL pointer, k outside [1, max_mz], steps < 1 or misaligned scratch; EIMS_ERR_STATE: no batch built.
 * Parameters and running statistics are not touched.  The plan is left as after eims_batch_build: a backward call
 * afterwards is refused until the next forward. */
int eims_attribute_peaks(eims_plan* p, const float* params, const float* bn_running, int32_t k, int32_t steps, int32_t* bins,
                         float* peak_prob, float* base_prob, float* ig, void* scratch, eims_stream_t stream);
/* The same in two parts, EIMS_BWD_HEAD then EIMS_BWD_GCN: after the head part the gradients of
 * the 10 spectrum_predictor tensors (the tail of the flat buffer, 84 % of its bytes) are final,
 * so a data-parallel caller can start reducing that bucket while the GCN layers are
 * differentiated (new functionality: the reference is single-GPU, GCN:63). */
int eims_backward_part(eims_plan* p, const float* params, const float* dprob, float* grads, int32_t part,
                       eims_stream_t stream);
/* metrics[8] (device): [0..2] += {sum_b row_loss/(B*M), mean_b row_cos, 1}; [4],[5] = this step's loss / cosine  - the per-step
 * `loss.item()` / `cos_sim.mean().item()` of GCN:436-437 without the host syncs; [6] += 1 for every step whose loss
 * was NaN / Inf (a guard the caller reads once per epoch together with the sums). */
int eims_metrics_accumulate(eims_plan* p, float* metrics, eims_stream_t stream);

/* One optimiser step: batch build + forward + loss + backward [+ AdamW when adam_m != NULL]. */
int eims_train_step(eims_plan* p, const eims_dataset* ds, const int32_t* mol_ids, int32_t num_graphs,
                    float* params, float* grads, float* adam_m, float* adam_v, float* bn_running,
                    int32_t loss_kind, const eims_step* s, float* metrics, eims_stream_t stream);
/* The same step on the batch eims_batch_build built last (forward + loss + backward [+ AdamW]).
 * The plan keeps two sets of batch tables and eims_batch_build always fills the set that the
 * work enqueued so far does not use, so the caller may build batch t+1 on a side stream while
 * step t runs (order the streams with events: the build of batch t+1 must wait for the end of
 * step t-1, step t+1 for the build).  targets / target_rows as in eims_loss. */
int eims_train_step_built(eims_plan* p, const float* targets, const int32_t* target_rows, float* params, float* grads,
                          float* adam_m, float* adam_v, float* bn_running, int32_t loss_kind, const eims_step* s,
                          float* metrics, eims_stream_t stream);
/* ---- one optimiser step as a replayable CUDA graph (new: the reference launches ~150 library kernels per step
 * from Python, GCN:410-431).  A captured graph freezes kernel parameters, so what changes from step to step - the
 * ids of the batch to build, the AdamW scalars of the one-cycle schedule (GCN:386-391, 429-431), the dropout keys,
 * the data-parallel sequence number - is kept in a small device "step block" (eims_step_block_bytes() bytes, caller
 * owned, 16-byte aligned).  eims_step_block_upload rewrites it with ONE tiny kernel that takes the values as launch
 * parameters (no host buffer has to stay alive); the *_indirect calls enqueue the same kernels as their plain
 * namesakes but those read the step block at execution time.  Usage: capture
 *     eims_train_step_built_indirect (main stream)  ||  eims_batch_build_indirect (side stream: next batch)
 * once per table set (the plan double-buffers the batch tables, so two graphs alternate), then per step:
 *     eims_step_block_upload(scalars of step t, ids of batch t+1) ; cudaGraphLaunch.
 * The target row of graph b is the molecule id it was built from (the ids K1 read). */
int64_t eims_step_block_bytes(void);
/* dev_block: room for one or more step blocks (bytes / eims_step_block_bytes() of them); NULL: indirect calls disabled.
 * A graph may hold SEVERAL consecutive steps (the launch gap between two graphs then amortises over them): give every
 * captured step its own block - eims_plan_select_step_block(k) before enqueueing step k - and fill blocks
 * [first, first + n) with one launch of eims_step_blocks_upload (n <= 16) before each replay. */
int eims_plan_set_step_block(eims_plan* p, void* dev_block, int64_t bytes);
int eims_plan_select_step_block(eims_plan* p, int32_t index);
int eims_step_block_upload(eims_plan* p, const eims_step* s, const int32_t* mol_ids, uint32_t dp_seq, eims_stream_t stream);
int eims_step_blocks_upload(eims_plan* p, const eims_step* steps, const int32_t* const* mol_ids, const uint32_t* dp_seq,
                            int32_t first, int32_t n, eims_stream_t stream);
int eims_batch_build_indirect(eims_plan* p, const eims_dataset* ds, int32_t num_graphs, eims_stream_t stream);
/* side_stream (may be NULL): a second stream for the work nothing on the step's chain waits for - the bias gradient
 * of the output layer and the AdamW update of the head tensors (84 % of the parameters) run there while the GCN layers
 * are differentiated; forked from and joined back into `stream` with events, i.e. graph edges under capture. */
int eims_train_step_built_indirect(eims_plan* p, const float* targets, float* params, float* grads, float* adam_m,
                                   float* adam_v, float* bn_running, int32_t loss_kind, float* metrics, eims_stream_t stream,
                                   eims_stream_t side_stream);
/* The same step in two parts for a caller that runs its own optimiser between them: part 1 = forward, loss and the
 * backward of the output head (the head gradients are final when it returns: a data-parallel caller starts exchanging
 * that bucket on a side stream), part 2 = the backward of the GraphConv layers.  No optimiser. */
int eims_train_step_built_indirect_part(eims_plan* p, const float* targets, float* params, float* grads, float* bn_running,
                                        int32_t loss_kind, float* metrics, int32_t part, eims_stream_t stream);

/* predict_spectrum (GCN:494-511) for a batch: batch build + eval forward + sigmoid. */
int eims_infer_batch(eims_plan* p, const eims_dataset* ds, const int32_t* mol_ids, int32_t num_graphs,
                     const float* params, const float* bn_running, float* prob_out, eims_stream_t stream);
/* Data-parallel optimiser step in one kernel (new functionality; the reference is single-GPU,
 * GCN:63): all-reduce of the flat gradient buffers + AdamW (GCN:429) + parameter broadcast over
 * NVLink / NVSwitch peer memory.  Rank r updates the slice [r*n/world, (r+1)*n/world) from the sum
 * of every rank's gradients (multimem.ld_reduce through the switch when `grads_multicast` != 0,
 * else peer loads) and stores it into every rank's parameter buffer (multimem.st / peer stores).
 * grad_ptrs / param_ptrs / signal_ptrs: `world` peer-mapped device addresses (host arrays) of
 * this step's gradient buffer, the parameter buffer and the signal pad (>= 512 bytes, zeroed
 * once) of every rank.  The call covers the float range [range_off, range_off + range_len) of the
 * flat buffers (range_off % 4 == 0, range_len a multiple of 4*world) so that a step can exchange
 * the head bucket early and the rest at the end; `bucket` (0..3) selects that range's signal rows
 * and m_slice / v_slice / ticket belong to the bucket (range_len/world floats; one zeroed word).
 * zero_buf: this rank's OTHER gradient buffer (gradients are double-buffered because peers read
 * them); its range is zeroed here.  seq: 1, 2, 3, ... the same on every rank.
 * s->grad_scale = 1/world.  `ticket` points at 4 zeroed words of the bucket: word 0 is the grid ticket, word 1 a
 * status word - a rank that waited longer than EIMS_DP_TIMEOUT_S (default 600 s) for a peer stores the sequence
 * number there and carries on (no trap: the context stays usable and the host reports the lost peer).
 * _blk: the same with the AdamW scalars and the sequence number read from a device step block (s, seq ignored when
 * step_block != NULL) so that the launch can sit inside a captured CUDA graph. */
int eims_dp_adamw_fused(int32_t rank, int32_t world, const uint64_t* grad_ptrs, const uint64_t* param_ptrs,
                        const uint64_t* signal_ptrs, uint64_t grads_multicast, uint64_t params_multicast,
                        float* m_slice, float* v_slice, float* zero_buf, int64_t range_off, int64_t range_len,
                        const eims_step* s, uint32_t seq, int32_t bucket, uint32_t* ticket, eims_stream_t stream);
int eims_dp_adamw_fused_blk(int32_t rank, int32_t world, const uint64_t* grad_ptrs, const uint64_t* param_ptrs,
                            const uint64_t* signal_ptrs, uint64_t grads_multicast, uint64_t params_multicast,
                            float* m_slice, float* v_slice, float* zero_buf, int64_t range_off, int64_t range_len,
                            const eims_step* s, uint32_t seq, int32_t bucket, uint32_t* ticket, const void* step_block,
                            eims_stream_t stream);

/* Per-stage device timing for the roofline report (bench.py): when enabled every kernel
 * launch of the plan is bracketed by CUDA events on the launching stream.  _read
 * synchronises, sums the elapsed ms and the bracket count per stage (eims_plan_num_stages()
 * entries, names from eims_plan_stage_name) and returns the number of kernels launched
 * since _profile was last called. */
int eims_plan_profile(eims_plan* p, int32_t enable);
int eims_plan_profile_read(eims_plan* p, float* stage_ms, int32_t* stage_launches, int32_t n_stages,
                           int64_t* total_launches);
int eims_plan_num_stages(void);
const char* eims_plan_stage_name(int32_t k);
/* Reads dims[] back (one small synchronous copy) and maps flags to error codes. */
int eims_plan_check(eims_plan* p, int32_t* num_nodes, int32_t* num_edges, eims_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* EIMS_B200_H_ */
