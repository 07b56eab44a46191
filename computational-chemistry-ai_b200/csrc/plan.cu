// The C ABI (include/eims_b200.h): parameter layout, workspace plan, and the whole-step
// orchestration  batch build -> GCNSpectrum.forward -> loss -> backward -> AdamW
// (reference: templates/ms-pred-gcn-eims-cupy.py:292-297, 354-376, 410-431).
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <type_traits>
#include <vector>

#include <nvtx3/nvToolsExt.h>  // header-only (dlopens the injection library when a profiler is attached)

#include "common.cuh"
#include "launchers.h"

using namespace eims;


namespace {

thread_local char g_err[512] = "";

constexpr int kMaxLayers = 16;  // GraphConv layers a plan can hold

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define EIMS_TRY(expr)                      \
  do {                                      \
    int _rc = (expr);                       \
    if (_rc != 0) return _rc < 0 ? fail(_rc, "%s failed (%d) at %s:%d", #expr, _rc, __FILE__, __LINE__) : _rc; \
  } while (0)

int check_launch(const char* what) {
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(EIMS_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
  }
  return 0;
}

int check_dims(const eims_dims* d) {
  if (!d) return fail(EIMS_ERR_ARG, "dims is NULL");
  if (d->node_feat_dim < 1 || d->node_feat_dim > 8) return fail(EIMS_ERR_ARG, "node_feat_dim must be in [1,8]");
  if (d->hidden_dim < 64 || d->hidden_dim % 64 || d->hidden_dim > 1024)
    return fail(EIMS_ERR_ARG, "hidden_dim must be a multiple of 64 in [64,1024]");
  if (d->num_gcn_layers < 1 || d->num_gcn_layers > kMaxLayers) return fail(EIMS_ERR_ARG, "num_gcn_layers must be in [1,16]");
  if (d->max_mz < 4 || d->max_mz % 4 || d->max_mz > 4096) return fail(EIMS_ERR_ARG, "max_mz must be a multiple of 4 in [4,4096]");
  if (d->pooling < 0 || d->pooling > 3) return fail(EIMS_ERR_ARG, "pooling must be one of EIMS_POOL_*");
  if (!(d->dropout >= 0.f && d->dropout < 1.f)) return fail(EIMS_ERR_ARG, "dropout must be in [0,1)");
  return 0;
}

// tensor sizes in model.parameters() order
std::vector<int64_t> param_sizes(const eims_dims* d) {
  const int64_t F = d->node_feat_dim, H = d->hidden_dim, M = d->max_mz, L = d->num_gcn_layers;
  const int64_t P = d->pooling == EIMS_POOL_COMBINED ? 2 * H : H;
  std::vector<int64_t> s;
  for (int l = 0; l < L; ++l) { s.push_back((l == 0 ? F : H) * H); s.push_back(H); }
  for (int l = 0; l < L; ++l) { s.push_back(H); s.push_back(H); }
  s.push_back(2 * H * P); s.push_back(2 * H); s.push_back(2 * H); s.push_back(2 * H);
  s.push_back(H * 2 * H); s.push_back(H); s.push_back(H); s.push_back(H);
  s.push_back(M * H); s.push_back(M);
  return s;
}

// The tables K1 writes for one batch.  The plan holds two sets of them (eims_plan::cur).
struct BatchTables {
  int *dims, *gptr, *eptr, *gid, *bids, *src, *dst, *rowptr, *col;
  float *norm, *x, *a0;
};

// The buffers of the bound workspace, carved by walk_workspace.
struct Workspace {
  BatchTables t[2];
  int *flags, *argmax;
  float* a[kMaxLayers];  // a_l for l >= 1 (layer 0 reads the batch table a0)
  float* wplanes;        // planes-capable plans only
  float *z[kMaxLayers], *bn_mean[kMaxLayers], *bn_invstd[kMaxLayers], *bn_scale[kMaxLayers], *bn_shift[kMaxLayers];
  float *bn_means2, *bn_partials, *readout, *zstat;
  float *u1, *u2, *logits, *dy2, *dy1, *dG;  // outputs of the split-K head GEMMs
  float *y1, *ln1, *y2, *ln2, *prob, *dlogits, *row_loss, *row_cos, *dh, *q, *da;
};

// Where a plan is in the calls on the batch built last; decides which calls it accepts.
enum class Phase {
  unbuilt,    // bound, no batch built yet
  built,      // batch built, or its training backward enqueued
  train_fwd,  // training forward enqueued
  loss_grad,  // ... and eims_loss(want_grad = 1): dlogits ready
  head_bwd,   // ... and the head part of the backward: the head gradients are final
  eval_fwd,   // eval-mode forward enqueued (eims_backward_feat may follow)
};

}  // namespace

struct eims_plan {
  eims_dims d;
  int Bc, Nc, Ec;  // capacities
  int gemm_backend;
  int64_t ws_bytes;
  bool bound;
  std::vector<int64_t> poff;  // parameter offsets
  Workspace ws{};
  int64_t head_zero_bytes = 0;  // bytes of the range [u1, end of dG) a training forward's layer-0 kernel zeroes
  Phase phase = Phase::unbuilt;
  bool after_train_fwd() const { return phase == Phase::train_fwd || phase == Phase::loss_grad || phase == Phase::head_bwd; }
  // per-stage CUDA-event profiling (bench.py's roofline pass) and launch accounting
  eims_peaks peak_targets{};  // targets as peak lists (eims_plan_set_peak_targets); peak_ptr == NULL: unset
  // BatchNorm-backward statistics of the layers below the top come out of the SpMM that writes their dh.  Beyond 256
  // columns the statistics variant of K2 needs 172 registers - one block per SM - and measured slower than K2 plus the
  // separate statistics pass: cfg 5, 0.99 + 0.02 ms against 0.38 + 0.43 ms per step.
  bool fuse_bn_bwd_stats = false;
  int batch_seq = 0;  // K1 sequence number (tags the zero-degree flag, see k1_build_kernel)
  bool prof = false;
  struct ProfRec { int stage; cudaEvent_t a, b; };
  std::vector<ProfRec> prof_recs;
  size_t prof_used = 0;
  int64_t launches = 0;
  eims_step last_step;
  // Planes path of the GraphConv products (csrc/gemm_tma.cu): a_l, q and the GraphConv weights exist as stacked tf32
  // hi / lo planes [2][rows][H] and the GEMMs are fed by the tensor-map copy engine.  planes_cap: the shapes allow it
  // (H a multiple of 256, <= 1024) and the workspace was sized for it; planes_on(): ... and the tensor-core backend is
  // selected.
  bool planes_cap = false;
  int64_t act_plane = 0;   // floats between the hi and the lo plane of a_l / q ( = rows_alloc * H )
  int64_t w_plane = 0;     // floats between the hi and the lo plane of the weight range [W_1 .. W_{L-1}]
  std::vector<TmaMap> maps;  // per layer l >= 1: a_l K-major, a_l MN-major, W_l MN-major (forward B), W_l K-major (dgrad B); then q K-major, q MN-major
  const TmaMap* map_a_k(int l) const { return &maps[4 * (l - 1) + 0]; }
  const TmaMap* map_a_mn(int l) const { return &maps[4 * (l - 1) + 1]; }
  const TmaMap* map_w_mn(int l) const { return &maps[4 * (l - 1) + 2]; }
  const TmaMap* map_w_k(int l) const { return &maps[4 * (l - 1) + 3]; }
  const TmaMap* map_q_k() const { return &maps[4 * (d.num_gcn_layers - 1) + 0]; }
  const TmaMap* map_q_mn() const { return &maps[4 * (d.num_gcn_layers - 1) + 1]; }
  // Measured on a B200 (profiles/r2_gemm_planes.md): with >= ~4 output tiles per SM (inference batches of 4096) the
  // persistent planes kernel hides every tile's epilogue under the next tile's main loop and runs at the MMA issue rate
  // (cfg 3: 6.9 -> 7.4 M molecules/s); at a training batch of 512 with hidden 256 a launch is ONE tile per SM, nothing
  // overlaps, and
  // what the planes cost (a second plane written by the producers, the weight split, twice the operand bytes from L2)
  // outweighs the faster main loop: 0.363 against 0.342 ms per step.  At hidden 1024 (cfg 5: 14 tiles per SM, K = 1024) the
  // planes kernel needs ~12 TB/s of operand bytes out of L2 to keep the tensor cores fed and gets ~7: 7.48 against 7.03 ms
  // per step - fp32 operands split in the kernel are half the bytes.  So: large batches at hidden <= 512 only, unless
  // eims_plan_set_gemm_planes(EIMS_PLANES_ON).
  bool planes_on() const {
    if (!(planes_cap && gemm_backend == EIMS_GEMM_TCGEN05 && gemm_tma_enabled() && !maps.empty())) return false;
    if (planes_mode >= 0) return planes_mode != 0;
    return d.hidden_dim <= 512 && (int64_t)((Nc + 127) / 128) * (d.hidden_dim / 256) >= 4 * 148;
  }
  int planes_mode = -1;  // eims_plan_set_gemm_planes
  int pool_dim() const { return d.pooling == EIMS_POOL_COMBINED ? 2 * d.hidden_dim : d.hidden_dim; }
  // rows of the shared-memory molecule tile of the aggregation / readout kernels: sized from the plan's own
  // atoms-per-molecule capacity (64 KB of tile: 64 rows x 256 columns or 128 rows x 128 columns); bigger molecules
  // take the gather path inside the same kernels
  int tile_rows() const { return (Nc + Bc - 1) / Bc <= 64 ? 64 : 128; }
  // The batch tables K1 writes exist twice ("name#0" / "name#1"): eims_batch_build always fills the
  // set the kernels enqueued so far do NOT use and makes it current for what is enqueued next, so
  // the next batch can be built on a side stream while the current step is still running.
  int cur = 0;
  const BatchTables& tab() const { return ws.t[cur]; }
  // Device step block (eims_plan_set_step_block) and the mode of the call being enqueued: `indirect` calls take
  // the batch's ids, the dropout keys and the AdamW scalars from it instead of from kernel parameters, so that
  // the launches can be captured into a CUDA graph once and replayed for every step.
  StepBlock* blk = nullptr;       // the block the next *_indirect calls bake in (eims_plan_select_step_block)
  StepBlock* blk_base = nullptr;  // the caller's array of blk_count blocks
  int blk_count = 0;
  bool indirect = false;
  // Side branch of a step (eims_train_step_built_indirect with a second stream): work that nothing on the chain
  // waits for - the output-layer bias gradient (colsum) and the AdamW update of the head tensors, 84 % of the
  // parameters - runs there while the GCN layers are differentiated on the main stream.  Fork / join are event
  // record / wait pairs, which stream capture turns into graph edges.
  cudaStream_t side = nullptr;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  int ensure_events() {
    for (auto& e : ev)
      if (!e && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return EIMS_ERR_CUDA;
    return 0;
  }
  DropCfg drop(float prob, uint64_t seed, int step, int site) const {
    DropCfg d = make_drop(prob, seed, step, site);
    if (indirect && blk && site >= 0 && site < kMaxDropSites) d.key_dev = &blk->drop_key[site];
    return d;
  }
  // parameter accessors (flat buffer)
  int64_t off_gcn_w(int l) const { return poff[2 * l]; }
  int64_t off_gcn_b(int l) const { return poff[2 * l + 1]; }
  int64_t off_bn_g(int l) const { return poff[2 * d.num_gcn_layers + 2 * l]; }
  int64_t off_bn_b(int l) const { return poff[2 * d.num_gcn_layers + 2 * l + 1]; }
  int64_t off_head(int k) const { return poff[4 * d.num_gcn_layers + k]; }  // 0..9
};

namespace {

int launch_gemm(int backend, const GemmProblem& q, cudaStream_t st) {
  return backend == EIMS_GEMM_FP32_SIMT ? launch_gemm_simt(q, st) : launch_gemm_tc(q, st);
}

// weight gradient + data gradient of one layer (both consume the same dy) in one launch
int gemm_pair(eims_plan* p, const GemmProblem& a, const GemmProblem& b, cudaStream_t st) {
  if (p->gemm_backend == EIMS_GEMM_FP32_SIMT) {
    if (int rc = launch_gemm_simt(a, st)) return rc;
    return launch_gemm_simt(b, st);
  }
  return launch_gemm_tc_pair(a, b, st);
}

// How eims_plan_buffer names a buffer: `name`, `name<l>` (per GraphConv layer), `name#<set>` (per batch-table set).
enum class Naming { plain, layer, set };

// Every workspace buffer in carve order, as f(name, naming, index, bytes, slot) with `slot` the typed pointer field the
// buffer is bound to.  Sizes are rounded up to 256 bytes, so in a 256-aligned workspace every buffer is 256-aligned.
// eims_plan_create sizes the workspace with it, eims_plan_bind carves it, eims_plan_buffer resolves names.
template <class Fn> void walk_workspace(eims_plan* p, Fn&& f) {
  Workspace& w = p->ws;
  const int64_t B = p->Bc, N = p->Nc, E = p->Ec, H = p->d.hidden_dim, F = p->d.node_feat_dim, M = p->d.max_mz;
  const int L = p->d.num_gcn_layers;
  const int64_t P = p->pool_dim();
  auto r = [](int64_t bytes) { return (bytes + 255) & ~(int64_t)255; };
  auto one = [&](const char* n, int64_t bytes, auto& slot) { f(n, Naming::plain, 0, r(bytes), slot); };
  auto layer = [&](const char* n, int l, int64_t bytes, auto& slot) { f(n, Naming::layer, l, r(bytes), slot); };
  auto sets = [&](const char* n, int64_t bytes, auto BatchTables::*m) {
    for (int k = 0; k < 2; ++k) f(n, Naming::set, k, r(bytes), w.t[k].*m);
  };
  sets("dims", 16 * 4, &BatchTables::dims); one("flags", 16 * 4, w.flags);
  sets("gptr", (B + 1) * 4, &BatchTables::gptr); sets("eptr", (B + 1) * 4, &BatchTables::eptr);
  sets("gid", N * 4, &BatchTables::gid); sets("bids", B * 4, &BatchTables::bids);
  sets("src", E * 4, &BatchTables::src); sets("dst", E * 4, &BatchTables::dst);
  sets("rowptr", (N + 1) * 4, &BatchTables::rowptr); sets("col", E * 4, &BatchTables::col);
  one("argmax", B * H * 4, w.argmax);
  sets("norm", N * 4, &BatchTables::norm); sets("x", N * F * 4, &BatchTables::x); sets("a0", N * F * 4, &BatchTables::a0);
  // a_l and q hold two planes (tf32 hi / lo) when the GraphConv GEMMs may take the planes path
  const int64_t act_bytes = p->planes_cap ? 2 * p->act_plane * 4 : N * H * 4;
  for (int l = 1; l < L; ++l) layer("a", l, act_bytes, w.a[l]);
  if (p->planes_cap) one("wplanes", 2 * p->w_plane * 4, w.wplanes);
  for (int l = 0; l < L; ++l) layer("z", l, N * H * 4, w.z[l]);
  for (int l = 0; l < L; ++l) {
    layer("bn_mean", l, H * 4, w.bn_mean[l]); layer("bn_invstd", l, H * 4, w.bn_invstd[l]);
    layer("bn_scale", l, H * 4, w.bn_scale[l]); layer("bn_shift", l, H * 4, w.bn_shift[l]);
  }
  one("bn_means2", 2 * H * 4, w.bn_means2);
  one("bn_partials", bn_scratch_floats(p->d.hidden_dim, p->Nc) * 4, w.bn_partials);
  one("readout", B * P * 4, w.readout);
  one("zstat", B * 2 * H * 4, w.zstat);  // per graph: raw column sums and raw arg-max values of the top layer (training)
  // outputs of the split-K head GEMMs, contiguous: a training forward zeroes the whole range once
  // (inside the layer-0 kernel) instead of one memset per GEMM, which would also break the
  // programmatic-dependent-launch chain six times per step
  one("u1", B * 2 * H * 4, w.u1); one("u2", B * H * 4, w.u2); one("logits", B * M * 4, w.logits);
  one("dy2", B * H * 4, w.dy2); one("dy1", B * 2 * H * 4, w.dy1); one("dG", B * P * 4, w.dG);
  one("y1", B * 2 * H * 4, w.y1); one("ln1", B * 2 * 4, w.ln1);
  one("y2", B * H * 4, w.y2); one("ln2", B * 2 * 4, w.ln2);
  one("prob", B * M * 4, w.prob); one("dlogits", B * M * 4, w.dlogits);
  one("row_loss", B * 4, w.row_loss); one("row_cos", B * 4, w.row_cos);
  one("dh", N * H * 4, w.dh); one("q", act_bytes, w.q); one("da", N * H * 4, w.da);
}

enum Stage {
  ST_K1 = 0, ST_LAYER0_FWD, ST_BN_STATS, ST_SPMM_FWD, ST_GEMM_GCN_FWD, ST_READOUT, ST_GEMM_HEAD_FWD, ST_LN_FWD, ST_LOSS,
  ST_METRICS, ST_GEMM_HEAD_WGRAD, ST_COLSUM, ST_GEMM_HEAD_DGRAD, ST_LN_BWD, ST_BN_BWD_STATS, ST_BN_BWD_APPLY, ST_GEMM_GCN_WGRAD,
  ST_GEMM_GCN_DGRAD, ST_SPMM_BWD, ST_LAYER0_WGRAD, ST_ADAMW, ST_ELEMENTWISE, ST_GEMM_HEAD_BWD, ST_GEMM_GCN_BWD, ST_COUNT
};
const char* kStageNames[ST_COUNT] = {
  "k1_batch_build", "layer0_fwd", "bn_stats", "spmm_fwd", "gemm_gcn_fwd", "readout", "gemm_head_fwd", "ln_fwd", "loss",
  "metrics", "gemm_head_wgrad", "colsum", "gemm_head_dgrad", "ln_bwd", "bn_bwd_stats", "bn_bwd_apply", "gemm_gcn_wgrad",
  "gemm_gcn_dgrad", "spmm_bwd", "layer0_wgrad", "adamw", "elementwise", "gemm_head_bwd", "gemm_gcn_bwd"};

// NVTX range per kernel class (stage) around its launches, for nsys / ncu timelines: EIMS_NVTX=1.  Off by default:
// the ranges are host-side calls on the launch path.
bool nvtx_on() {
  static int on = -1;
  if (on < 0) { const char* e = getenv("EIMS_NVTX"); on = (e && e[0] == '1') ? 1 : 0; }
  return on != 0;
}

void prof_begin(eims_plan* p, int stage, int nkernels, cudaStream_t st) {
  p->launches += nkernels;
  if (nvtx_on()) nvtxRangePushA(kStageNames[stage]);
  if (!p->prof) return;
  if (p->prof_used == p->prof_recs.size()) {
    eims_plan::ProfRec r;
    r.stage = stage;
    cudaEventCreate(&r.a);
    cudaEventCreate(&r.b);
    p->prof_recs.push_back(r);
  }
  p->prof_recs[p->prof_used].stage = stage;
  cudaEventRecord(p->prof_recs[p->prof_used].a, st);
}
void prof_end(eims_plan* p, cudaStream_t st) {
  if (nvtx_on()) nvtxRangePop();
  if (!p->prof) return;
  cudaEventRecord(p->prof_recs[p->prof_used].b, st);
  ++p->prof_used;
}
// resets the "sizes may be read before the grid-dependency wait" flag however the function is left
struct EarlyDimsScope {
  explicit EarlyDimsScope(int v) { dims_early_ref() = v; }
  ~EarlyDimsScope() { dims_early_ref() = 0; }
};

#define STAGE(id, nk, expr)          \
  do {                               \
    prof_begin(p, id, nk, st);       \
    EIMS_TRY(expr);                  \
    prof_end(p, st);                 \
  } while (0)

}  // namespace

#pragma GCC visibility push(default)
extern "C" {

int eims_version(void) { return 100; }
const char* eims_last_error(void) { return g_err; }

int eims_device_check(void) {
  int dev = 0;
  cudaDeviceProp prop;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&prop, dev) != cudaSuccess)
    return fail(EIMS_ERR_CUDA, "no CUDA device");
  if (prop.major != 10) return fail(EIMS_ERR_CUDA, "device is sm_%d%d; this library is built for sm_100a only", prop.major, prop.minor);
  return 0;
}

int64_t eims_param_count(const eims_dims* d) {
  if (check_dims(d)) return -1;
  int64_t n = 0;
  for (int64_t s : param_sizes(d)) n += s;
  return n;
}
int eims_param_num_tensors(const eims_dims* d) { return check_dims(d) ? -1 : 4 * d->num_gcn_layers + 10; }
int eims_param_layout(const eims_dims* d, int64_t* offsets, int32_t n_entries) {
  EIMS_TRY(check_dims(d));
  auto s = param_sizes(d);
  if (!offsets || n_entries != (int)s.size() + 1) return fail(EIMS_ERR_ARG, "offsets must have %d entries", (int)s.size() + 1);
  int64_t o = 0;
  for (size_t k = 0; k < s.size(); ++k) { offsets[k] = o; o += s[k]; }
  offsets[s.size()] = o;
  return 0;
}

// ------------------------------------------------------------------ stand-alone kernels
int eims_csr_build(const eims_dataset* ds, const int32_t* mol_ids, int32_t num_graphs, int32_t node_feat_dim,
                   int32_t max_nodes, int32_t max_edges, int32_t* gptr, int32_t* eptr, int32_t* gid, int32_t* src,
                   int32_t* dst, int32_t* rowptr, int32_t* col, float* norm, float* x, int32_t* dims,
                   eims_stream_t stream) {
  if (!ds || num_graphs < 0) return fail(EIMS_ERR_ARG, "bad dataset / num_graphs");
  if (cudaMemsetAsync(dims + DIM_ZERO_DEG, 0, sizeof(int32_t), (cudaStream_t)stream) != cudaSuccess)
    return fail(EIMS_ERR_CUDA, "cudaMemsetAsync failed");
  EIMS_TRY(launch_csr_build(ds, mol_ids, num_graphs, node_feat_dim, max_nodes, max_edges, gptr, eptr, gid, src, dst,
                            rowptr, col, norm, x, dims, (cudaStream_t)stream));
  return check_launch("eims_csr_build");
}

int eims_spmm_norm(const int32_t* dims, const int32_t* rowptr, const int32_t* col, const float* norm, const float* h,
                   int32_t width, const float* bn_scale, const float* bn_shift, float drop_p, uint64_t seed,
                   int32_t step, int32_t site, int32_t out_scale_norm, float* out, int32_t max_nodes,
                   eims_stream_t stream) {
  EIMS_TRY(launch_spmm_norm(dims, rowptr, col, norm, h, width, bn_scale, bn_shift, make_drop(drop_p, seed, step, site),
                            out_scale_norm ? 1 : 0, out, max_nodes, (cudaStream_t)stream));
  return check_launch("eims_spmm_norm");
}

int eims_spmm_norm_mol(const int32_t* dims, const int32_t* gptr, const int32_t* rowptr, const int32_t* col, const float* norm,
                       const float* h, int32_t width, const float* bn_scale, const float* bn_shift, float drop_p, uint64_t seed,
                       int32_t step, int32_t site, int32_t out_scale_norm, float* out, int32_t max_nodes, int32_t max_graphs,
                       int32_t tile_rows, eims_stream_t stream) {
  if (!gptr || tile_rows < 1 || tile_rows > 128 || width % 128) return fail(EIMS_ERR_ARG, "gptr / tile_rows in [1,128] / width %% 128");
  (void)max_nodes;
  EIMS_TRY(launch_spmm_mol(dims, gptr, rowptr, col, norm, h, width, bn_scale, bn_shift, make_drop(drop_p, seed, step, site),
                           out_scale_norm ? 1 : 0, out, max_graphs, tile_rows, (cudaStream_t)stream, nullptr));
  return check_launch("eims_spmm_norm_mol");
}

int eims_gemm(int32_t backend, const float* A, int32_t lda, int32_t a_mn_major, const float* B, int32_t ldb,
              int32_t b_mn_major, float* C, int32_t ldc, int32_t M, int32_t N, int32_t K, const int32_t* m_dev,
              const int32_t* k_dev, const float* row_scale, const float* bias, int32_t relu, int32_t accumulate,
              eims_stream_t stream) {
  EIMS_TRY(launch_gemm(backend, GemmProblem{.A = A, .lda = lda, .a_mn = a_mn_major, .B = B, .ldb = ldb, .b_mn = b_mn_major,
                                             .C = C, .ldc = ldc, .M = M, .N = N, .K = K, .m_dev = m_dev, .k_dev = k_dev,
                                             .row_scale = row_scale, .bias = bias, .relu = relu,
                                             .accumulate = static_cast<GemmAcc>(accumulate)},
                       (cudaStream_t)stream));
  return check_launch("eims_gemm");
}

// stand-alone form of the planes GEMM: split both operands of each problem into scratch, encode the maps, launch
static int64_t planes_rows(const eims_gemm_problem* q, bool b) {
  return b ? (q->b_mn_major ? q->K : q->N) : (q->a_mn_major ? q->K : q->M);
}
int64_t eims_gemm_planes_scratch_bytes(const eims_gemm_problem* p0, const eims_gemm_problem* p1) {
  int64_t bytes = 0;
  for (const eims_gemm_problem* q : {p0, p1})
    if (q) bytes += 2 * 4 * (planes_rows(q, false) * q->lda + planes_rows(q, true) * q->ldb) + 512;
  return bytes;
}
int eims_gemm_planes(const eims_gemm_problem* p0, const eims_gemm_problem* p1, void* scratch, int64_t scratch_bytes,
                     eims_stream_t stream) {
  if (!p0 || !scratch) return fail(EIMS_ERR_ARG, "problem / scratch is NULL");
  if (scratch_bytes < eims_gemm_planes_scratch_bytes(p0, p1)) return fail(EIMS_ERR_ARG, "scratch too small");
  if (reinterpret_cast<uintptr_t>(scratch) & 255) return fail(EIMS_ERR_ARG, "scratch must be 256-byte aligned");
  if (!gemm_tma_enabled()) return fail(EIMS_ERR_STATE, "the planes GEMM is unavailable (no cuTensorMapEncodeTiled)");
  cudaStream_t st = (cudaStream_t)stream;
  TmaMap maps[4];
  GemmTmaProblem gp[2];
  char* c = reinterpret_cast<char*>(scratch);
  int n = 0;
  for (const eims_gemm_problem* q : {p0, p1}) {
    if (!q) continue;
    if (!q->A || !q->B || !q->C || (q->lda & 3) || (q->ldb & 3)) return fail(EIMS_ERR_ARG, "operands NULL or lda / ldb not a multiple of 4");
    const float* src[2] = {q->A, q->B};
    const int64_t rows[2] = {planes_rows(q, false), planes_rows(q, true)};
    const int ld[2] = {q->lda, q->ldb}, mn[2] = {q->a_mn_major, q->b_mn_major};
    const int cols[2] = {q->a_mn_major ? q->M : q->K, q->b_mn_major ? q->N : q->K};
    for (int o = 0; o < 2; ++o) {
      const int64_t plane = rows[o] * ld[o];
      float* hi = reinterpret_cast<float*>(c);
      EIMS_TRY(launch_split_planes(src[o], hi, hi + plane, plane, st, false));
      EIMS_TRY(tma_make_map(&maps[2 * n + o], hi, plane, (int)rows[o], cols[o], ld[o], o ? kTmaBRows : 128, mn[o]));
      c += ((2 * 4 * plane + 255) & ~(int64_t)255);
    }
    gp[n] = GemmTmaProblem{.ta = &maps[2 * n], .tb = &maps[2 * n + 1], .C = q->C, .ldc = q->ldc, .a_mn = q->a_mn_major,
                           .b_mn = q->b_mn_major, .M = q->M, .N = q->N, .K = q->K, .m_dev = q->m_dev, .k_dev = q->k_dev,
                           .row_scale = q->row_scale, .bias = q->bias, .relu = q->relu, .red = q->accumulate ? 1 : 0};
    if (!gemm_tma_supports(gp[n])) return fail(EIMS_ERR_ARG, "shape not supported by the planes GEMM (N %% 256, ldc %% 4, K <= 512 unless split-K)");
    ++n;
  }
  EIMS_TRY(launch_gemm_tma(&gp[0], n > 1 ? &gp[1] : nullptr, st));
  return check_launch("eims_gemm_planes");
}

int64_t eims_bn_scratch_floats(int32_t width, int32_t max_nodes) { return bn_scratch_floats(width, max_nodes); }

int eims_bn_stats(const int32_t* dims, const float* z, int32_t width, const float* gamma, const float* beta,
                  float* running_mean, float* running_var, float* mean, float* invstd, float* scale, float* shift,
                  float* partials, int32_t max_nodes, eims_stream_t stream) {
  EIMS_TRY(launch_bn_stats(dims, z, width, gamma, beta, running_mean, running_var, mean, invstd, scale, shift, partials,
                           max_nodes, (cudaStream_t)stream));
  return check_launch("eims_bn_stats");
}

int eims_readout(const int32_t* dims, const int32_t* gptr, const float* z, int32_t width, const float* bn_scale,
                 const float* bn_shift, int32_t pooling, float* out, int32_t* argmax, int32_t max_graphs,
                 eims_stream_t stream) {
  EIMS_TRY(launch_readout(dims, gptr, z, width, bn_scale, bn_shift, pooling, out, argmax, max_graphs, (cudaStream_t)stream));
  return check_launch("eims_readout");
}

int eims_loss_mse_cos(const int32_t* dims, const float* logits, const float* targets, const int32_t* target_rows,
                      int32_t max_mz, int32_t loss_kind, float* prob, float* dlogits, float* row_loss, float* row_cos,
                      int32_t max_graphs, eims_stream_t stream) {
  EIMS_TRY(launch_loss(dims, logits, targets, target_rows, max_mz, loss_kind, prob, dlogits, row_loss, row_cos,
                       max_graphs, (cudaStream_t)stream));
  return check_launch("eims_loss_mse_cos");
}

int eims_peaks_to_spectrum(const eims_peaks* pk, const int32_t* rows, int32_t num_rows, int32_t max_mz, float* out,
                           eims_stream_t stream) {
  if (!pk) return fail(EIMS_ERR_ARG, "peaks is NULL");
  if (max_mz < 1 || max_mz > 4096) return fail(EIMS_ERR_ARG, "max_mz must be in [1,4096]");
  EIMS_TRY(launch_peaks_to_spectrum(pk, rows, num_rows, max_mz, out, (cudaStream_t)stream));
  return check_launch("eims_peaks_to_spectrum");
}

int eims_topk_peaks(const float* spectra, int32_t num_rows, int32_t max_mz, int32_t k, int32_t* idx_out, float* val_out,
                    eims_stream_t stream) {
  if (!spectra || !idx_out) return fail(EIMS_ERR_ARG, "spectra / idx_out is NULL");
  if (max_mz < 1 || max_mz > 4096 || k < 1 || k > max_mz) return fail(EIMS_ERR_ARG, "need 1 <= k <= max_mz <= 4096");
  EIMS_TRY(launch_topk_peaks(spectra, num_rows, max_mz, k, idx_out, val_out, (cudaStream_t)stream));
  return check_launch("eims_topk_peaks");
}

int eims_adamw_flat(float* p, float* g, float* m, float* v, int64_t n, const eims_step* s, eims_stream_t stream) {
  EIMS_TRY(launch_adamw(p, g, m, v, n, s, (cudaStream_t)stream));
  return check_launch("eims_adamw_flat");
}

int eims_dropout_mask(float drop_p, uint64_t seed, int32_t step, int32_t site, int32_t rows, int32_t width, float* out,
                      eims_stream_t stream) {
  EIMS_TRY(launch_dropout_mask(make_drop(drop_p, seed, step, site), rows, width, out, (cudaStream_t)stream));
  return check_launch("eims_dropout_mask");
}

// ------------------------------------------------------------------ plan
int eims_plan_create(const eims_dims* d, int32_t max_graphs, int32_t max_nodes, int32_t max_edges, eims_plan** out) {
  EIMS_TRY(check_dims(d));
  if (!out || max_graphs < 1 || max_nodes < 1 || max_edges < 0) return fail(EIMS_ERR_ARG, "bad capacities");
  eims_plan* p = new eims_plan();
  p->d = *d;
  p->Bc = max_graphs; p->Nc = max_nodes; p->Ec = max_edges > 0 ? max_edges : 1;
  p->gemm_backend = EIMS_GEMM_TCGEN05;
  p->fuse_bn_bwd_stats = d->hidden_dim <= 256;
  p->ws_bytes = 0; p->bound = false;
  memset(&p->last_step, 0, sizeof(p->last_step));
  auto s = param_sizes(d);
  int64_t o = 0;
  for (int64_t v : s) { p->poff.push_back(o); o += v; }
  p->poff.push_back(o);
  const int64_t N = p->Nc, H = d->hidden_dim, L = d->num_gcn_layers;
  // a_l and q hold two planes (tf32 hi / lo) when the GraphConv GEMMs may take the planes path; rows padded to 32
  p->planes_cap = gemm_tma_enabled() && H % 256 == 0 && H <= 1024 && L > 1;
  p->act_plane = ((N + 31) & ~(int64_t)31) * H;
  p->w_plane = p->planes_cap ? (p->off_gcn_w(L - 1) + H * H - p->off_gcn_w(1)) : 0;
  // The layer-0 kernel of a training forward zeroes [u1, end of dG) as one range: the six split-K head outputs must
  // follow one another in the carve order, with nothing in between.
  const Workspace& w = p->ws;
  const void* const head[] = {&w.u1, &w.u2, &w.logits, &w.dy2, &w.dy1, &w.dG};
  int next = 0;  // head[next] is the head output expected next
  bool contiguous = true;
  walk_workspace(p, [&](const char*, Naming, int, int64_t bytes, auto& slot) {
    if (next < 6 && static_cast<const void*>(&slot) == head[next]) {
      ++next;
      p->head_zero_bytes += bytes;
    } else if (next > 0 && next < 6) {
      contiguous = false;
    }
    p->ws_bytes += bytes;
  });
  if (next != 6 || !contiguous) {
    delete p;
    return fail(EIMS_ERR_STATE, "workspace layout: the head outputs u1 .. dG are not contiguous");
  }
  *out = p;
  return 0;
}

int eims_plan_destroy(eims_plan* p) {
  if (p) for (auto& r : p->prof_recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  if (p) for (auto& e : p->ev) if (e) cudaEventDestroy(e);
  delete p;
  return 0;
}
int64_t eims_plan_workspace_bytes(const eims_plan* p) { return p ? p->ws_bytes : -1; }

int eims_plan_bind(eims_plan* p, void* workspace, int64_t bytes) {
  if (!p || !workspace) return fail(EIMS_ERR_ARG, "plan / workspace is NULL");
  if (bytes < p->ws_bytes) return fail(EIMS_ERR_ARG, "workspace too small: %lld < %lld", (long long)bytes, (long long)p->ws_bytes);
  if (reinterpret_cast<uintptr_t>(workspace) & 255) return fail(EIMS_ERR_ARG, "workspace must be 256-byte aligned");
  Workspace& w = p->ws;
  // counters / flags / dims start at zero (the ticket counter in bn_partials must be 0)
  const void* const zeroed[] = {&w.t[0].dims, &w.t[1].dims, &w.flags, &w.bn_partials};
  char* c = reinterpret_cast<char*>(workspace);
  cudaError_t e = cudaSuccess;
  walk_workspace(p, [&](const char*, Naming, int, int64_t bytes, auto& slot) {
    slot = reinterpret_cast<std::remove_reference_t<decltype(slot)>>(c);
    for (const void* z : zeroed)
      if (z == static_cast<const void*>(&slot) && e == cudaSuccess) e = cudaMemset(c, 0, bytes);
    c += bytes;
  });
  if (e != cudaSuccess) return fail(EIMS_ERR_CUDA, "cudaMemset failed: %s", cudaGetErrorString(cudaGetLastError()));
  p->maps.clear();
  if (p->planes_cap) {
    const int L = p->d.num_gcn_layers, H = p->d.hidden_dim;
    const int rows = (int)(p->act_plane / H);
    p->maps.resize(4 * (L - 1) + 2);
    int rc = 0;
    for (int l = 1; l < L && !rc; ++l) {
      const float* wl = w.wplanes + (p->off_gcn_w(l) - p->off_gcn_w(1));
      rc = tma_make_map(&p->maps[4 * (l - 1) + 0], w.a[l], p->act_plane, rows, H, H, 128, 0);
      if (!rc) rc = tma_make_map(&p->maps[4 * (l - 1) + 1], w.a[l], p->act_plane, rows, H, H, 128, 1);
      if (!rc) rc = tma_make_map(&p->maps[4 * (l - 1) + 2], wl, p->w_plane, H, H, H, kTmaBRows, 1);
      if (!rc) rc = tma_make_map(&p->maps[4 * (l - 1) + 3], wl, p->w_plane, H, H, H, kTmaBRows, 0);
    }
    if (!rc) rc = tma_make_map(&p->maps[4 * (L - 1) + 0], w.q, p->act_plane, rows, H, H, 128, 0);
    if (!rc) rc = tma_make_map(&p->maps[4 * (L - 1) + 1], w.q, p->act_plane, rows, H, H, 128, 1);
    if (rc) p->maps.clear();  // the encoder refused: the in-kernel-split GEMMs take over (planes_on() is false)
  }
  p->bound = true;
  p->phase = Phase::unbuilt;
  return 0;
}

int eims_plan_set_gemm_backend(eims_plan* p, int32_t backend) {
  if (!p || (backend != EIMS_GEMM_TCGEN05 && backend != EIMS_GEMM_FP32_SIMT)) return fail(EIMS_ERR_ARG, "bad backend");
  p->gemm_backend = backend;
  return 0;
}

int eims_plan_set_gemm_planes(eims_plan* p, int32_t mode) {
  if (!p || mode < -1 || mode > 1) return fail(EIMS_ERR_ARG, "mode must be one of EIMS_PLANES_*");
  if (mode == 1 && !(p->planes_cap && (!p->bound || !p->maps.empty())))
    return fail(EIMS_ERR_STATE, "the planes GEMM needs hidden_dim %% 256 == 0, >= 2 GCN layers and cuTensorMapEncodeTiled");
  p->planes_mode = mode;
  return 0;
}

int eims_plan_buffer(eims_plan* p, const char* name, void** ptr, int64_t* bytes) {
  if (!p || !p->bound || !name) return fail(EIMS_ERR_STATE, "plan not bound");
  bool found = false;
  walk_workspace(p, [&](const char* base, Naming how, int k, int64_t n, auto& slot) {
    if (found) return;
    char full[32];
    if (how == Naming::plain) snprintf(full, sizeof(full), "%s", base);
    else snprintf(full, sizeof(full), how == Naming::layer ? "%s%d" : "%s#%d", base, k);
    // a bare batch-table name means the current set
    if (strcmp(name, full) != 0 && !(how == Naming::set && k == p->cur && strcmp(name, base) == 0)) return;
    found = true;
    if (ptr) *ptr = slot;
    if (bytes) *bytes = n;
  });
  if (!found) return fail(EIMS_ERR_ARG, "no workspace buffer named '%s'", name);
  return 0;
}

static int batch_build_impl(eims_plan* p, const eims_dataset* ds, const int32_t* mol_ids, int32_t num_graphs,
                            eims_stream_t stream, bool indirect) {
  if (!p || !p->bound) return fail(EIMS_ERR_STATE, "plan not bound");
  if (indirect && !p->blk) return fail(EIMS_ERR_STATE, "no step block set (eims_plan_set_step_block)");
  if (!ds || num_graphs < 0) return fail(EIMS_ERR_ARG, "bad dataset / num_graphs");
  if (num_graphs > p->Bc) return fail(EIMS_ERR_CAPACITY, "num_graphs %d exceeds plan max_graphs %d", num_graphs, p->Bc);
  cudaStream_t st = (cudaStream_t)stream;
  p->cur ^= 1;  // build into the other set of batch tables; later calls use it
  if (p->batch_seq >= 0x7ffffff0) {  // sequence wrap: forget the old zero-degree tag
    for (const BatchTables& t : p->ws.t)
      if (cudaMemsetAsync(t.dims + DIM_ZERO_DEG, 0, sizeof(int), st) != cudaSuccess)
        return fail(EIMS_ERR_CUDA, "cudaMemsetAsync failed");
    p->batch_seq = 0;
  }
  ++p->batch_seq;
  const BatchTables& t = p->tab();
  STAGE(ST_K1, num_graphs > 1024 ? 2 : 1, launch_csr_build(ds, mol_ids, num_graphs, p->d.node_feat_dim, p->Nc, p->Ec, t.gptr, t.eptr,
                            t.gid, t.src, t.dst, t.rowptr, t.col, t.norm, t.x, t.dims, st, t.a0, p->batch_seq,
                            indirect ? p->blk : nullptr, t.bids));
  p->phase = Phase::built;
  return check_launch("eims_batch_build");
}

int eims_batch_build(eims_plan* p, const eims_dataset* ds, const int32_t* mol_ids, int32_t num_graphs,
                     eims_stream_t stream) {
  return batch_build_impl(p, ds, mol_ids, num_graphs, stream, false);
}

int eims_batch_build_indirect(eims_plan* p, const eims_dataset* ds, int32_t num_graphs, eims_stream_t stream) {
  return batch_build_impl(p, ds, nullptr, num_graphs, stream, true);
}

int eims_plan_set_step_block(eims_plan* p, void* dev_block, int64_t bytes) {
  if (!p) return fail(EIMS_ERR_ARG, "plan is NULL");
  if (dev_block && (bytes < (int64_t)sizeof(StepBlock) || (reinterpret_cast<uintptr_t>(dev_block) & 15)))
    return fail(EIMS_ERR_ARG, "step block needs %d bytes, 16-byte aligned", (int)sizeof(StepBlock));
  p->blk_base = p->blk = reinterpret_cast<StepBlock*>(dev_block);
  p->blk_count = dev_block ? (int)(bytes / (int64_t)sizeof(StepBlock)) : 0;
  return 0;
}
int64_t eims_step_block_bytes(void) { return (int64_t)sizeof(StepBlock); }

int eims_plan_select_step_block(eims_plan* p, int32_t index) {
  if (!p || !p->blk_base) return fail(EIMS_ERR_STATE, "no step block set (eims_plan_set_step_block)");
  if (index < 0 || index >= p->blk_count) return fail(EIMS_ERR_ARG, "step block %d outside [0, %d)", index, p->blk_count);
  p->blk = p->blk_base + index;
  return 0;
}

static StepBlock make_step_block(const eims_plan* p, const eims_step* s, const int32_t* mol_ids, uint32_t dp_seq) {
  StepBlock v{};
  v.ids = mol_ids;
  v.adam = make_adam_k(s);
  const int sites = p->d.num_gcn_layers + 2;
  for (int k = 0; k < sites && k < kMaxDropSites; ++k) v.drop_key[k] = drop_key(s->seed, s->step, k);
  v.dp_seq = dp_seq;
  v.k1_seq = 1 + (s->step & 0x3fffffff);
  return v;
}

int eims_step_blocks_upload(eims_plan* p, const eims_step* steps, const int32_t* const* mol_ids, const uint32_t* dp_seq,
                            int32_t first, int32_t n, eims_stream_t stream) {
  if (!p || !p->blk_base) return fail(EIMS_ERR_STATE, "no step block set (eims_plan_set_step_block)");
  if (!steps || !mol_ids || n < 1 || n > kStepPack || first < 0 || first + n > p->blk_count)
    return fail(EIMS_ERR_ARG, "need 1 <= n <= %d blocks inside [0, %d)", kStepPack, p->blk_count);
  StepBlockPack pack{};
  for (int k = 0; k < n; ++k) {
    if (steps[k].step < 1) return fail(EIMS_ERR_ARG, "step < 1");
    pack.b[k] = make_step_block(p, steps + k, mol_ids[k], dp_seq ? dp_seq[k] : 0u);
  }
  EIMS_TRY(launch_step_blocks_store(pack, p->blk_base + first, n, (cudaStream_t)stream));
  return check_launch("eims_step_blocks_upload");
}

int eims_step_block_upload(eims_plan* p, const eims_step* s, const int32_t* mol_ids, uint32_t dp_seq, eims_stream_t stream) {
  if (!p || !p->blk) return fail(EIMS_ERR_STATE, "no step block set (eims_plan_set_step_block)");
  if (!s || s->step < 1) return fail(EIMS_ERR_ARG, "step scalars are NULL / step < 1");
  return eims_step_blocks_upload(p, s, &mol_ids, &dp_seq, (int32_t)(p->blk - p->blk_base), 1, stream);
}

int eims_forward(eims_plan* p, const float* params, float* bn_running, int32_t training, const eims_step* s,
                 eims_stream_t stream) {
  if (!p || !p->bound) return fail(EIMS_ERR_STATE, "plan not bound");
  if (p->phase == Phase::unbuilt) return fail(EIMS_ERR_STATE, "eims_forward before eims_batch_build");
  if (!params || !bn_running) return fail(EIMS_ERR_ARG, "params / bn_running is NULL");
  cudaStream_t st = (cudaStream_t)stream;
  const eims_dims& d = p->d;
  const int H = d.hidden_dim, F = d.node_feat_dim, L = d.num_gcn_layers, M = d.max_mz, P = p->pool_dim();
  const BatchTables& t = p->tab();
  const Workspace& w = p->ws;
  const int* dims = t.dims;
  const float drop_p = (training && d.dropout > 0.f) ? d.dropout : 0.f;
  const uint64_t seed = s ? s->seed : 0;
  const int step = s ? s->step : 0;
  if (s) p->last_step = *s;
  auto bn = [&](int l) -> int {
    float* rm = bn_running + (int64_t)l * 2 * H;
    float* rv = rm + H;
    if (training)
      return launch_bn_stats(dims, w.z[l], H, params + p->off_bn_g(l), params + p->off_bn_b(l), rm, rv, w.bn_mean[l],
                             w.bn_invstd[l], w.bn_scale[l], w.bn_shift[l], w.bn_partials, p->Nc, st);
    return launch_bn_eval_coeffs(params + p->off_bn_g(l), params + p->off_bn_b(l), rm, rv, H, w.bn_scale[l], w.bn_shift[l],
                                 st, w.bn_mean[l], w.bn_invstd[l]);
  };
  auto fuse = [&](int l) {
    float* rm = bn_running + (int64_t)l * 2 * H;
    return BnFuse{reinterpret_cast<double*>(w.bn_partials + 16), reinterpret_cast<unsigned int*>(w.bn_partials),
                  params + p->off_bn_g(l), params + p->off_bn_b(l), rm, rm + H, w.bn_mean[l], w.bn_invstd[l], w.bn_scale[l],
                  w.bn_shift[l], H};
  };
  {  // layer 0: dense transform of K1's 6-wide aggregate, BatchNorm statistics fused when training
    BnFuse bf{};
    if (training) bf = fuse(0);
    // training: the kernel also zeroes the split-K head outputs, the range [u1, end of dG) (contiguous: eims_plan_create)
    float* zero = training ? w.u1 : nullptr;
    STAGE(ST_LAYER0_FWD, 1, launch_layer0_fwd(dims, t.norm, t.a0, F, params + p->off_gcn_w(0), params + p->off_gcn_b(0),
                               H, w.z[0], p->Nc, st, training ? &bf : nullptr, zero, p->head_zero_bytes / 16));
    if (!training) STAGE(ST_BN_STATS, 1, bn(0));
  }
  // every launch from here on is at least two kernels after the batch build: sizes before the grid-dependency wait
  EarlyDimsScope early_scope(1);
  const bool planes = p->planes_on();
  if (planes)  // hi / lo planes of the GraphConv weights W_1 .. W_{L-1} (one pass over the range that holds them)
    STAGE(ST_ELEMENTWISE, 1, launch_split_planes(params + p->off_gcn_w(1), w.wplanes, w.wplanes + p->w_plane, p->w_plane, st, true));
  for (int l = 1; l < L; ++l) {
    // training on the tensor-core path: the BatchNorm statistics of z_l come out of the GEMM epilogue
    const bool fuse_bn = training && p->gemm_backend == EIMS_GEMM_TCGEN05;
    BnFuse bf{};
    if (fuse_bn) bf = fuse(l);
    STAGE(ST_SPMM_FWD, 1, launch_spmm_norm(dims, t.rowptr, t.col, t.norm, w.z[l - 1], H, w.bn_scale[l - 1], w.bn_shift[l - 1],
                              p->drop(drop_p, seed, step, l - 1), 0, w.a[l], p->Nc, st, nullptr, t.gptr, p->Bc,
                              p->tile_rows(), planes ? p->act_plane : 0));
    if (planes) {
      GemmTmaProblem fw{.ta = p->map_a_k(l), .tb = p->map_w_mn(l), .C = w.z[l], .ldc = H, .b_mn = 1, .M = p->Nc, .N = H,
                        .K = H, .m_dev = dims + DIM_N, .row_scale = t.norm, .bias = params + p->off_gcn_b(l), .relu = 1,
                        .bn = fuse_bn ? &bf : nullptr};
      STAGE(ST_GEMM_GCN_FWD, 1, launch_gemm_tma(&fw, nullptr, st));
    } else {
      STAGE(ST_GEMM_GCN_FWD, 1, launch_gemm(p->gemm_backend,
            GemmProblem{.A = w.a[l], .lda = H, .B = params + p->off_gcn_w(l), .ldb = H, .b_mn = 1, .C = w.z[l], .ldc = H,
                        .M = p->Nc, .N = H, .K = H, .m_dev = dims + DIM_N, .row_scale = t.norm,
                        .bias = params + p->off_gcn_b(l), .relu = 1, .bn = fuse_bn ? &bf : nullptr}, st));
    }
    if (!fuse_bn) STAGE(ST_BN_STATS, 1, bn(l));
  }
  // The 512-row head GEMMs cannot fill 148 SMs with output tiles, so in training they split K and
  // accumulate with float atomics (summation order varies in the last bit run to run); eval-mode
  // forwards keep plain stores and are bit-reproducible.
  const GemmAcc head_acc = training ? kGemmStoreSplitZeroed : kGemmStore;  // C zeroed by the layer-0 kernel
  STAGE(ST_READOUT, 1, launch_readout(dims, t.gptr, w.z[L - 1], H, w.bn_scale[L - 1], w.bn_shift[L - 1], d.pooling, w.readout,
                          w.argmax, p->Bc, st, training ? w.zstat : nullptr, training ? w.bn_mean[L - 1] : nullptr));
  STAGE(ST_GEMM_HEAD_FWD, 1, launch_gemm(p->gemm_backend,
        GemmProblem{.A = w.readout, .lda = P, .B = params + p->off_head(0), .ldb = P, .C = w.u1, .ldc = 2 * H, .M = p->Bc,
                    .N = 2 * H, .K = P, .m_dev = dims + DIM_B, .bias = params + p->off_head(1), .accumulate = head_acc}, st));
  STAGE(ST_LN_FWD, 1, launch_ln_fwd(dims, w.u1, 2 * H, params + p->off_head(2), params + p->off_head(3),
                         p->drop(drop_p, seed, step, L), w.y1, w.ln1, p->Bc, st));
  STAGE(ST_GEMM_HEAD_FWD, 1, launch_gemm(p->gemm_backend,
        GemmProblem{.A = w.y1, .lda = 2 * H, .B = params + p->off_head(4), .ldb = 2 * H, .C = w.u2, .ldc = H, .M = p->Bc,
                    .N = H, .K = 2 * H, .m_dev = dims + DIM_B, .bias = params + p->off_head(5), .accumulate = head_acc}, st));
  STAGE(ST_LN_FWD, 1, launch_ln_fwd(dims, w.u2, H, params + p->off_head(6), params + p->off_head(7),
                         p->drop(drop_p, seed, step, L + 1), w.y2, w.ln2, p->Bc, st));
  STAGE(ST_GEMM_HEAD_FWD, 1, launch_gemm(p->gemm_backend,
        GemmProblem{.A = w.y2, .lda = H, .B = params + p->off_head(8), .ldb = H, .C = w.logits, .ldc = M, .M = p->Bc, .N = M,
                    .K = H, .m_dev = dims + DIM_B, .bias = params + p->off_head(9), .accumulate = head_acc}, st));
  p->phase = training ? Phase::train_fwd : Phase::eval_fwd;
  return check_launch("eims_forward");
}

int eims_sigmoid(eims_plan* p, eims_stream_t stream) {
  if (!p || !p->bound) return fail(EIMS_ERR_STATE, "plan not bound");
  cudaStream_t st = (cudaStream_t)stream;
  STAGE(ST_ELEMENTWISE, 1, launch_sigmoid(p->tab().dims, p->ws.logits, p->d.max_mz, p->ws.prob, p->Bc, (cudaStream_t)stream));
  return check_launch("eims_sigmoid");
}

int eims_plan_set_peak_targets(eims_plan* p, const eims_peaks* pk) {
  if (!p) return fail(EIMS_ERR_ARG, "plan is NULL");
  if (pk && !(pk->peak_ptr && pk->mz && pk->intensity)) return fail(EIMS_ERR_ARG, "peak_ptr / mz / intensity is NULL");
  p->peak_targets = pk ? *pk : eims_peaks{};
  return 0;
}

static int loss_impl(eims_plan* p, const float* targets, const int32_t* target_rows, int32_t loss_kind, int32_t want_grad,
                     float* metrics, eims_stream_t stream, const eims_peaks* peaks = nullptr) {
  if (!p || !p->bound) return fail(EIMS_ERR_STATE, "plan not bound");
  if (!targets && !peaks && p->peak_targets.peak_ptr) peaks = &p->peak_targets;
  if (!targets && !peaks) return fail(EIMS_ERR_ARG, "targets is NULL (and no peak-list targets are set)");
  cudaStream_t st = (cudaStream_t)stream;
  // after a training forward, never right after a batch build (nor after an eval forward, which may follow one)
  EarlyDimsScope early_scope(p->after_train_fwd() ? 1 : 0);
  // metrics != NULL: the last block of the loss kernel also folds the row terms into the running
  // metrics (flags[0] is its ticket), which saves the separate one-block launch
  const Workspace& w = p->ws;
  STAGE(ST_LOSS, 1, launch_loss(p->tab().dims, w.logits, targets, target_rows, p->d.max_mz, loss_kind, w.prob,
                       want_grad ? w.dlogits : nullptr, w.row_loss, w.row_cos, p->Bc,
                       (cudaStream_t)stream, metrics, reinterpret_cast<unsigned int*>(w.flags), peaks));
  if (want_grad && p->phase == Phase::train_fwd) p->phase = Phase::loss_grad;
  return check_launch("eims_loss");
}

int eims_loss(eims_plan* p, const float* targets, const int32_t* target_rows, int32_t loss_kind, int32_t want_grad,
              eims_stream_t stream) {
  return loss_impl(p, targets, target_rows, loss_kind, want_grad, nullptr, stream);
}

// The data-only eval backward of eims_attribute_peaks: the gradient of prob[r, bins[r]] summed over the graphs, down to
// the atom features only, weighted into the integrated gradients (launch_ig_feat_accum).
struct PeakGrad {
  const int* bins;  // m_r per graph
  float weight;     // 1 / steps
  bool first;       // the first path point: ig = weight * dx (later: ig += weight * dx)
  const float* x;   // the last path point: the atom features ig is then multiplied by (else NULL)
};

// The backward of the forward enqueued last, for every public entry point: the training step's (eval = false, dfeat
// NULL: eims_backward, eims_backward_part), eims_backward_feat's (either mode, optionally down to the atom features) and
// eims_attribute_peaks' (pg != NULL: eval mode, no parameter gradients - grads is not touched - and into dfeat = ig).
// The callers have checked the plan's state.
static int backward_impl(eims_plan* p, const float* params, const float* dprob, float* grads, int32_t part, float* dfeat,
                         bool eval, cudaStream_t st, const PeakGrad* pg = nullptr) {
  EarlyDimsScope early_scope(1);  // backward always follows a forward (training or eval)
  const eims_dims& d = p->d;
  const int H = d.hidden_dim, F = d.node_feat_dim, L = d.num_gcn_layers, M = d.max_mz, P = p->pool_dim();
  const BatchTables& t = p->tab();
  const Workspace& w = p->ws;
  const int* dims = t.dims;
  // eval mode: no dropout, BatchNorm is the affine map of the running statistics (bn_mean<l> / bn_invstd<l> hold them,
  // written by the eval forward), so its backward has no batch-statistics terms: the two column means the apply pass
  // subtracts stay zero (the statistics passes get means == NULL)
  const float drop_p = (!eval && d.dropout > 0.f) ? d.dropout : 0.f;
  const float drop_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
  float* means2 = eval ? nullptr : w.bn_means2;
  // the head data gradients: a training forward's layer-0 kernel zeroed dy2 / dy1 / dG (split-K allowed); an eval
  // forward zeroes nothing, so there they are plain stores
  const GemmAcc head_acc = eval ? kGemmStore : kGemmStoreSplitZeroed;
  const uint64_t seed = p->last_step.seed;
  const int step = p->last_step.step;
  const bool planes = p->planes_on();  // as in the forward that produced a_l (the backend must not change in between)
  const int* dB = dims + DIM_B;
  if (pg) {
    // ---- head, data gradients only: dy2 gathered from W3's row m_r, LayerNorm backward without its parameter
    // gradients, and the two remaining products as plain data-gradient GEMMs
    STAGE(ST_ELEMENTWISE, 1, launch_peak_head_dgrad(dims, w.logits, M, pg->bins, params + p->off_head(8), H, w.dy2, p->Bc, st));
    STAGE(ST_LN_BWD, 1, launch_ln_dgrad(dims, w.u2, w.y2, w.dy2, H, params + p->off_head(6), w.ln2, w.dy2, p->Bc, st));
    STAGE(ST_GEMM_HEAD_DGRAD, 1, launch_gemm(p->gemm_backend,
          GemmProblem{.A = w.dy2, .lda = H, .B = params + p->off_head(4), .ldb = 2 * H, .b_mn = 1, .C = w.dy1, .ldc = 2 * H,
                      .M = p->Bc, .N = 2 * H, .K = H, .m_dev = dB}, st));
    STAGE(ST_LN_BWD, 1, launch_ln_dgrad(dims, w.u1, w.y1, w.dy1, 2 * H, params + p->off_head(2), w.ln1, w.dy1, p->Bc, st));
    STAGE(ST_GEMM_HEAD_DGRAD, 1, launch_gemm(p->gemm_backend,
          GemmProblem{.A = w.dy1, .lda = 2 * H, .B = params + p->off_head(0), .ldb = P, .b_mn = 1, .C = w.dG, .ldc = P,
                      .M = p->Bc, .N = P, .K = 2 * H, .m_dev = dB}, st));
  }
  if (eval && !pg) {
    if (cudaMemsetAsync(w.bn_means2, 0, 2 * (size_t)H * sizeof(float), st) != cudaSuccess)
      return fail(EIMS_ERR_CUDA, "cudaMemsetAsync failed");
    // prob of this forward (an eval forward leaves only the logits; eims_sigmoid may not have run)
    STAGE(ST_ELEMENTWISE, 1, launch_sigmoid(dims, w.logits, M, w.prob, p->Bc, st));
  }
  if (part != EIMS_BWD_GCN && !pg) {
  if (dprob) STAGE(ST_ELEMENTWISE, 1, launch_dprob_to_dlogits(dims, w.prob, dprob, M, w.dlogits, p->Bc, st));
  float* dl = w.dlogits;
  // ---- head (GCN:341-352 backwards)
  if (p->side) {  // fork: the bias gradient of the output layer is needed by AdamW only
    if (cudaEventRecord(p->ev[0], st) != cudaSuccess || cudaStreamWaitEvent(p->side, p->ev[0], 0) != cudaSuccess)
      return fail(EIMS_ERR_CUDA, "side-branch fork failed: %s", cudaGetErrorString(cudaGetLastError()));
    prof_begin(p, ST_COLSUM, 1, p->side);
    EIMS_TRY(launch_colsum(dims, DIM_B, dl, M, M, grads + p->off_head(9), p->Bc, p->side));
    prof_end(p, p->side);
  } else {
    STAGE(ST_COLSUM, 1, launch_colsum(dims, DIM_B, dl, M, M, grads + p->off_head(9), p->Bc, st));
  }
  STAGE(ST_GEMM_HEAD_BWD, p->gemm_backend == EIMS_GEMM_TCGEN05 ? 1 : 2, gemm_pair(p,
        GemmProblem{.A = dl, .lda = M, .a_mn = 1, .B = w.y2, .ldb = H, .b_mn = 1, .C = grads + p->off_head(8), .ldc = H,
                    .M = M, .N = H, .K = p->Bc, .k_dev = dB, .accumulate = kGemmAdd},
        GemmProblem{.A = dl, .lda = M, .B = params + p->off_head(8), .ldb = H, .b_mn = 1, .C = w.dy2, .ldc = H, .M = p->Bc,
                    .N = H, .K = M, .m_dev = dB, .accumulate = head_acc}, st));
  // LayerNorm backward also leaves the bias gradient of the Linear in front of it (column sums of du)
  STAGE(ST_LN_BWD, 1, launch_ln_bwd(dims, w.u2, w.y2, w.dy2, H, params + p->off_head(6), w.ln2, drop_scale,
                         w.dy2, grads + p->off_head(6), grads + p->off_head(7), grads + p->off_head(5), p->Bc, st));
  STAGE(ST_GEMM_HEAD_BWD, p->gemm_backend == EIMS_GEMM_TCGEN05 ? 1 : 2, gemm_pair(p,
        GemmProblem{.A = w.dy2, .lda = H, .a_mn = 1, .B = w.y1, .ldb = 2 * H, .b_mn = 1, .C = grads + p->off_head(4),
                    .ldc = 2 * H, .M = H, .N = 2 * H, .K = p->Bc, .k_dev = dB, .accumulate = kGemmAdd},
        GemmProblem{.A = w.dy2, .lda = H, .B = params + p->off_head(4), .ldb = 2 * H, .b_mn = 1, .C = w.dy1, .ldc = 2 * H,
                    .M = p->Bc, .N = 2 * H, .K = H, .m_dev = dB, .accumulate = head_acc}, st));
  STAGE(ST_LN_BWD, 1, launch_ln_bwd(dims, w.u1, w.y1, w.dy1, 2 * H, params + p->off_head(2), w.ln1,
                         drop_scale, w.dy1, grads + p->off_head(2), grads + p->off_head(3), grads + p->off_head(1), p->Bc, st));
  STAGE(ST_GEMM_HEAD_BWD, p->gemm_backend == EIMS_GEMM_TCGEN05 ? 1 : 2, gemm_pair(p,
        GemmProblem{.A = w.dy1, .lda = 2 * H, .a_mn = 1, .B = w.readout, .ldb = P, .b_mn = 1, .C = grads + p->off_head(0),
                    .ldc = P, .M = 2 * H, .N = P, .K = p->Bc, .k_dev = dB, .accumulate = kGemmAdd},
        GemmProblem{.A = w.dy1, .lda = 2 * H, .B = params + p->off_head(0), .ldb = P, .b_mn = 1, .C = w.dG, .ldc = P,
                    .M = p->Bc, .N = P, .K = 2 * H, .m_dev = dB, .accumulate = head_acc}, st));
  if (!eval) p->phase = Phase::head_bwd;  // head gradients final (the data-parallel reducer may start on that bucket)
  }
  if (part == EIMS_BWD_HEAD) return check_launch("eims_backward_part");
  // ---- GCN layers, last to first (GCN:358-363 backwards)
  for (int l = L - 1; l >= 0; --l) {
    // the top layer's dh is the readout backward of dG, computed on the fly, and its BatchNorm-backward statistics come
    // from per-graph quantities; the layers below read the dh that the backward SpMM of the layer above wrote, and their
    // statistics pass rides on that SpMM when fuse_bn_bwd_stats (see below)
    const bool from_readout = (l == L - 1);
    const float* dh_in = from_readout ? nullptr : w.dh;
    if (pg) {
      // eval-mode BatchNorm backward: the statistics passes only produce dgamma / dbeta; layer 0 leaves q_0 plain
      STAGE(ST_BN_BWD_APPLY, 1, launch_bn_dgrad_apply(dims, dh_in, w.dG, t.gid, t.gptr, w.argmax, d.pooling, w.z[l], H,
                                   w.bn_mean[l], w.bn_invstd[l], params + p->off_bn_g(l), t.norm, w.q, p->Nc, st,
                                   (planes && l > 0) ? p->act_plane : 0));
      if (l > 0 && planes) {
        GemmTmaProblem dg{.ta = p->map_q_k(), .tb = p->map_w_k(l), .C = w.da, .ldc = H, .M = p->Nc, .N = H, .K = H,
                          .m_dev = dims + DIM_N};
        STAGE(ST_GEMM_GCN_DGRAD, 1, launch_gemm_tma(&dg, nullptr, st));
      } else if (l > 0) {
        STAGE(ST_GEMM_GCN_DGRAD, 1, launch_gemm(p->gemm_backend,
              GemmProblem{.A = w.q, .lda = H, .B = params + p->off_gcn_w(l), .ldb = H, .C = w.da, .ldc = H, .M = p->Nc,
                          .N = H, .K = H, .m_dev = dims + DIM_N}, st));
      }
      if (l > 0) {
        STAGE(ST_SPMM_BWD, 1, launch_spmm_norm(dims, t.rowptr, t.col, t.norm, w.da, H, nullptr, nullptr, make_drop(0.f, 0, 0, 0),
                                  1, w.dh, p->Nc, st, nullptr, t.gptr, p->Bc, p->tile_rows()));
      } else {
        STAGE(ST_GEMM_GCN_DGRAD, 1, launch_layer0_dgrad(dims, w.q, H, params + p->off_gcn_w(0), F, w.da, p->Nc, st));
        STAGE(ST_SPMM_BWD, 1, launch_ig_feat_accum(dims, t.rowptr, t.col, t.norm, w.da, F, pg->weight, pg->first, pg->x,
                                     dfeat, p->Nc, st));
      }
      continue;
    }
    if (from_readout) {
      if (eval)  // the per-graph sums a training readout leaves in zstat, about the running mean
        STAGE(ST_BN_BWD_STATS, 1, launch_bn_eval_zstat(dims, t.gptr, w.z[l], H, w.bn_mean[l], w.argmax, d.pooling, w.zstat,
                                     p->Bc, st));
      STAGE(ST_BN_BWD_STATS, 1, launch_bn_bwd_stats_top(dims, w.dG, w.zstat, t.gptr, d.pooling, H, w.bn_mean[l],
                                   w.bn_invstd[l], grads + p->off_bn_g(l), grads + p->off_bn_b(l), means2,
                                   w.bn_partials, p->Bc, st));
    } else if (!p->fuse_bn_bwd_stats) {
      STAGE(ST_BN_BWD_STATS, 1, launch_bn_bwd_stats(dims, dh_in, w.z[l], H, w.bn_mean[l], w.bn_invstd[l],
                                   grads + p->off_bn_g(l), grads + p->off_bn_b(l), means2, w.bn_partials, p->Nc, st));
    }
    STAGE(ST_BN_BWD_APPLY, 1, launch_bn_bwd_apply(dims, dh_in, w.dG, t.gid, t.gptr, w.argmax, d.pooling,
                                 w.z[l], H, w.bn_mean[l], w.bn_invstd[l], params + p->off_bn_g(l),
                                 t.norm, grads + p->off_gcn_b(l), w.bn_means2, w.q, p->Nc, st,
                                 l == 0 ? t.a0 : nullptr, F, l == 0 ? grads + p->off_gcn_w(0) : nullptr,
                                 (planes && l > 0) ? p->act_plane : 0, l == 0 && dfeat));
    if (l > 0 && planes) {
      // one persistent launch: data gradient tiles (stores) + weight gradient k-slices (red.add), balanced on the device
      GemmTmaProblem dg{.ta = p->map_q_k(), .tb = p->map_w_k(l), .C = w.da, .ldc = H, .M = p->Nc, .N = H, .K = H,
                        .m_dev = dims + DIM_N};
      GemmTmaProblem wg{.ta = p->map_a_mn(l), .tb = p->map_q_mn(), .C = grads + p->off_gcn_w(l), .ldc = H, .a_mn = 1, .b_mn = 1,
                        .M = H, .N = H, .K = p->Nc, .k_dev = dims + DIM_N, .red = 1};
      STAGE(ST_GEMM_GCN_BWD, 1, launch_gemm_tma(&dg, &wg, st));
    } else if (l > 0) {
      STAGE(ST_GEMM_GCN_BWD, p->gemm_backend == EIMS_GEMM_TCGEN05 ? 1 : 2, gemm_pair(p,
            GemmProblem{.A = w.a[l], .lda = H, .a_mn = 1, .B = w.q, .ldb = H, .b_mn = 1, .C = grads + p->off_gcn_w(l), .ldc = H,
                        .M = H, .N = H, .K = p->Nc, .k_dev = dims + DIM_N, .accumulate = kGemmAdd},
            GemmProblem{.A = w.q, .lda = H, .B = params + p->off_gcn_w(l), .ldb = H, .C = w.da, .ldc = H, .M = p->Nc, .N = H,
                        .K = H, .m_dev = dims + DIM_N}, st));
    }
    if (l > 0) {
      BnBwdFuse bf{w.z[l - 1], w.bn_mean[l - 1], w.bn_invstd[l - 1],
                   reinterpret_cast<double*>(w.bn_partials + 16), reinterpret_cast<unsigned int*>(w.bn_partials),
                   grads + p->off_bn_g(l - 1), grads + p->off_bn_b(l - 1), means2};
      STAGE(ST_SPMM_BWD, 1, launch_spmm_norm(dims, t.rowptr, t.col, t.norm, w.da, H, nullptr, nullptr,
                                p->drop(drop_p, seed, step, l - 1), 1, w.dh, p->Nc, st,
                                p->fuse_bn_bwd_stats ? &bf : nullptr, t.gptr, p->Bc, p->tile_rows()));
    } else if (dfeat) {
      // layer 0: dW0 came out of the apply pass above, which also left q_0 in q; da and dh are free here
      STAGE(ST_GEMM_GCN_DGRAD, 1, launch_layer0_dgrad(dims, w.q, H, params + p->off_gcn_w(0), F, w.da, p->Nc, st));
      STAGE(ST_SPMM_BWD, 1, launch_feat_grad(dims, t.rowptr, t.col, t.norm, w.da, F, dfeat, p->Nc, st));
    }  // l == 0 without dfeat: q_0 is never materialised
  }
  if (!eval) p->phase = Phase::built;
  return check_launch("eims_backward");
}

int eims_backward_part(eims_plan* p, const float* params, const float* dprob, float* grads, int32_t part,
                       eims_stream_t stream) {
  if (!p || !p->bound) return fail(EIMS_ERR_STATE, "plan not bound");
  if (part < EIMS_BWD_ALL || part > EIMS_BWD_GCN) return fail(EIMS_ERR_ARG, "part must be one of EIMS_BWD_*");
  if (!p->after_train_fwd()) return fail(EIMS_ERR_STATE, "eims_backward needs a training-mode eims_forward first");
  if (part == EIMS_BWD_GCN) {
    if (p->phase != Phase::head_bwd) return fail(EIMS_ERR_STATE, "EIMS_BWD_GCN needs EIMS_BWD_HEAD first");
  } else if (!dprob && p->phase != Phase::loss_grad) {
    return fail(EIMS_ERR_STATE, "eims_backward without dprob needs eims_loss(want_grad=1) first");
  }
  if (!params || !grads) return fail(EIMS_ERR_ARG, "params / grads is NULL");
  return backward_impl(p, params, dprob, grads, part, nullptr, false, (cudaStream_t)stream);
}

int eims_backward(eims_plan* p, const float* params, const float* dprob, float* grads, eims_stream_t stream) {
  return eims_backward_part(p, params, dprob, grads, EIMS_BWD_ALL, stream);
}

int eims_backward_feat(eims_plan* p, const float* params, const float* dprob, float* grads, float* dfeat,
                       eims_stream_t stream) {
  if (!p || !p->bound) return fail(EIMS_ERR_STATE, "plan not bound");
  const bool eval = p->phase == Phase::eval_fwd;
  if (!eval) {
    if (!p->after_train_fwd())
      return fail(EIMS_ERR_STATE, "eims_backward_feat needs an eims_forward of the batch built last (and no backward since)");
    if (p->phase == Phase::head_bwd) return fail(EIMS_ERR_STATE, "eims_backward_feat after EIMS_BWD_HEAD");
    if (!dprob && p->phase != Phase::loss_grad) return fail(EIMS_ERR_STATE, "eims_backward_feat without dprob needs eims_loss(want_grad=1) first");
  } else if (!dprob) {
    return fail(EIMS_ERR_ARG, "dprob is NULL: an eval-mode backward needs the gradient w.r.t. the spectrum");
  }
  if (!params || !grads) return fail(EIMS_ERR_ARG, "params / grads is NULL");
  return backward_impl(p, params, dprob, grads, EIMS_BWD_ALL, dfeat, eval, (cudaStream_t)stream);
}

int eims_attribute_peaks(eims_plan* p, const float* params, const float* bn_running, int32_t k, int32_t steps, int32_t* bins,
                         float* peak_prob, float* base_prob, float* ig, void* scratch, eims_stream_t stream) {
  if (!p || !p->bound) return fail(EIMS_ERR_STATE, "plan not bound");
  if (p->phase == Phase::unbuilt) return fail(EIMS_ERR_STATE, "eims_attribute_peaks before eims_batch_build");
  if (!params || !bn_running || !bins || !peak_prob || !base_prob || !ig || !scratch)
    return fail(EIMS_ERR_ARG, "params / bn_running / bins / peak_prob / base_prob / ig / scratch is NULL");
  if (k < 1 || k > p->d.max_mz || steps < 1) return fail(EIMS_ERR_ARG, "need 1 <= k <= max_mz and steps >= 1");
  if (reinterpret_cast<uintptr_t>(scratch) & 255) return fail(EIMS_ERR_ARG, "scratch must be 256-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int F = p->d.node_feat_dim, M = p->d.max_mz;
  const BatchTables& t = p->tab();
  const Workspace& w = p->ws;
  float* params_f = const_cast<float*>(params);
  float* running = const_cast<float*>(bn_running);  // an eval forward only reads it
  // scratch: the unscaled a0 [N, F], then the top-k table of the spectra at alpha = 1 (bins [B, k], values [B, k])
  auto r = [](int64_t bytes) { return (bytes + 255) & ~(int64_t)255; };
  char* c = reinterpret_cast<char*>(scratch);
  float* a0 = reinterpret_cast<float*>(c);
  int* top_idx = reinterpret_cast<int*>(c + r((int64_t)p->Nc * F * 4));
  float* top_val = reinterpret_cast<float*>(c + r((int64_t)p->Nc * F * 4) + r((int64_t)p->Bc * k * 4));
  STAGE(ST_ELEMENTWISE, 1, launch_feat_scale(t.dims, t.a0, F, 1.f, a0, p->Nc, st));
  // alpha = 1: the predicted spectra and their peaks
  EIMS_TRY(eims_forward(p, params_f, running, 0, nullptr, stream));
  STAGE(ST_ELEMENTWISE, 1, launch_sigmoid(t.dims, w.logits, M, w.prob, p->Bc, st));
  STAGE(ST_ELEMENTWISE, 1, launch_topk_peaks(w.prob, p->Bc, M, k, top_idx, top_val, st));
  STAGE(ST_ELEMENTWISE, 1, launch_peak_select(t.dims, top_idx, top_val, k, bins, peak_prob, p->Bc, st));
  // alpha = 0: the baseline
  STAGE(ST_ELEMENTWISE, 1, launch_feat_scale(t.dims, a0, F, 0.f, t.a0, p->Nc, st));
  EIMS_TRY(eims_forward(p, params_f, running, 0, nullptr, stream));
  STAGE(ST_ELEMENTWISE, 1, launch_peak_prob(t.dims, w.logits, M, bins, base_prob, p->Bc, st));
  // the path: a0 = A D (alpha x) = alpha a0, so the forward at alpha X starts from the scaled aggregate
  for (int s = 0; s < steps; ++s) {
    STAGE(ST_ELEMENTWISE, 1, launch_feat_scale(t.dims, a0, F, ((float)s + 0.5f) / (float)steps, t.a0, p->Nc, st));
    EIMS_TRY(eims_forward(p, params_f, running, 0, nullptr, stream));
    const PeakGrad pg{bins, 1.f / (float)steps, s == 0, s == steps - 1 ? t.x : nullptr};
    EIMS_TRY(backward_impl(p, params, nullptr, nullptr, EIMS_BWD_ALL, ig, true, st, &pg));
  }
  STAGE(ST_ELEMENTWISE, 1, launch_feat_scale(t.dims, a0, F, 1.f, t.a0, p->Nc, st));  // the batch tables as K1 left them
  p->phase = Phase::built;
  return check_launch("eims_attribute_peaks");
}

int eims_metrics_accumulate(eims_plan* p, float* metrics, eims_stream_t stream) {
  if (!p || !p->bound || !metrics) return fail(EIMS_ERR_STATE, "plan not bound / metrics NULL");
  cudaStream_t st = (cudaStream_t)stream;
  STAGE(ST_METRICS, 1, launch_metrics(p->tab().dims, p->ws.row_loss, p->ws.row_cos, p->d.max_mz, metrics, (cudaStream_t)stream));
  return check_launch("eims_metrics_accumulate");
}

// One training step on the batch built last, as every eims_train_step* entry point enqueues it.
struct StepCall {
  const float* targets;         // dense target rows; NULL: `peaks`, else the plan's peak-list targets
  const eims_peaks* peaks;
  const int32_t* target_rows;   // direct calls only: an indirect step reads the rows K1 took from the step block
  float *params, *grads, *adam_m, *adam_v, *bn_running;  // AdamW runs when adam_m and adam_v are both set
  int32_t loss_kind;
  const eims_step* s;           // direct: the step's scalars; NULL: indirect, scalars and dropout keys from the step block
  float* metrics;
  int32_t part;                 // EIMS_BWD_ALL; EIMS_BWD_HEAD: forward, loss, head backward; EIMS_BWD_GCN: the rest
  cudaStream_t st, side;        // side (indirect only): output-layer bias gradient and the head's AdamW
};

// forward -> loss (+ metrics) -> backward [-> AdamW].  The plan's per-call mode (indirect, side) is set here only and
// must not leak out of this function.
static int enqueue_step(eims_plan* p, const StepCall& c) {
  if (!p || !p->bound) return fail(EIMS_ERR_STATE, "plan not bound");
  const cudaStream_t st = c.st, side = c.side == c.st ? nullptr : c.side;
  if (side && p->ensure_events()) return fail(EIMS_ERR_CUDA, "cudaEventCreate failed");
  const eims_stream_t stream = (eims_stream_t)st;
  const bool indirect = !c.s;
  struct Mode {
    eims_plan* p;
    ~Mode() { p->indirect = false; p->side = nullptr; }
  } mode{p};
  p->indirect = indirect;
  p->side = side;
  if (c.part != EIMS_BWD_GCN) {
    const eims_step dummy{};  // indirect: seed / step are not used, the dropout keys come from the step block
    EIMS_TRY(eims_forward(p, c.params, c.bn_running, 1, indirect ? &dummy : c.s, stream));
    EIMS_TRY(loss_impl(p, c.targets, indirect ? p->tab().bids : c.target_rows, c.loss_kind, 1, c.metrics, stream,
                       c.targets ? nullptr : c.peaks));
  }
  if (c.part != EIMS_BWD_ALL) return eims_backward_part(p, c.params, nullptr, c.grads, c.part, stream);
  const bool adam = c.adam_m && c.adam_v;
  const StepBlock* blk = indirect ? p->blk : nullptr;
  const int64_t P = p->poff.back();
  if (!side || !adam) {
    EIMS_TRY(eims_backward(p, c.params, nullptr, c.grads, stream));
    if (adam) STAGE(ST_ADAMW, 1, launch_adamw(c.params, c.grads, c.adam_m, c.adam_v, P, c.s, st, blk));
    if (side) {  // join the colsum branch
      if (cudaEventRecord(p->ev[1], side) != cudaSuccess || cudaStreamWaitEvent(st, p->ev[1], 0) != cudaSuccess)
        return fail(EIMS_ERR_CUDA, "side-branch join failed");
    }
    return 0;
  }
  // head part on the main stream (its bias-gradient colsum on the side branch), then
  //   side: AdamW of the head range, as soon as the head gradients are final   ||   main: GCN layers backward
  const int64_t split = p->off_head(0) & ~(int64_t)3;   // [0, split) GraphConv + BatchNorm tensors, [split, P) the head
  EIMS_TRY(eims_backward_part(p, c.params, nullptr, c.grads, EIMS_BWD_HEAD, stream));
  if (cudaEventRecord(p->ev[2], st) != cudaSuccess || cudaStreamWaitEvent(side, p->ev[2], 0) != cudaSuccess)
    return fail(EIMS_ERR_CUDA, "side-branch fork failed");
  prof_begin(p, ST_ADAMW, 1, side);
  EIMS_TRY(launch_adamw(c.params + split, c.grads + split, c.adam_m + split, c.adam_v + split, P - split, c.s, side, blk));
  prof_end(p, side);
  if (cudaEventRecord(p->ev[1], side) != cudaSuccess) return fail(EIMS_ERR_CUDA, "cudaEventRecord failed");
  p->side = nullptr;  // the GCN part has nothing for the side branch
  EIMS_TRY(eims_backward_part(p, c.params, nullptr, c.grads, EIMS_BWD_GCN, stream));
  if (split > 0) STAGE(ST_ADAMW, 1, launch_adamw(c.params, c.grads, c.adam_m, c.adam_v, split, c.s, st, blk));
  if (cudaStreamWaitEvent(st, p->ev[1], 0) != cudaSuccess) return fail(EIMS_ERR_CUDA, "side-branch join failed");
  return 0;
}

int eims_train_step(eims_plan* p, const eims_dataset* ds, const int32_t* mol_ids, int32_t num_graphs, float* params,
                    float* grads, float* adam_m, float* adam_v, float* bn_running, int32_t loss_kind,
                    const eims_step* s, float* metrics, eims_stream_t stream) {
  if (!s) return fail(EIMS_ERR_ARG, "step scalars are NULL");
  if (!ds || (!ds->targets && !ds->peaks)) return fail(EIMS_ERR_ARG, "training needs dataset targets (dense rows or peak lists)");
  EIMS_TRY(eims_batch_build(p, ds, mol_ids, num_graphs, stream));
  return enqueue_step(p, {ds->targets, ds->peaks, mol_ids, params, grads, adam_m, adam_v, bn_running, loss_kind, s, metrics,
                          EIMS_BWD_ALL, (cudaStream_t)stream, nullptr});
}

int eims_train_step_built(eims_plan* p, const float* targets, const int32_t* target_rows, float* params, float* grads,
                          float* adam_m, float* adam_v, float* bn_running, int32_t loss_kind, const eims_step* s,
                          float* metrics, eims_stream_t stream) {
  if (!s) return fail(EIMS_ERR_ARG, "step scalars are NULL");
  if (!targets && !(p && p->peak_targets.peak_ptr)) return fail(EIMS_ERR_ARG, "training needs target spectra");
  return enqueue_step(p, {targets, nullptr, target_rows, params, grads, adam_m, adam_v, bn_running, loss_kind, s, metrics,
                          EIMS_BWD_ALL, (cudaStream_t)stream, nullptr});
}

int eims_train_step_built_indirect(eims_plan* p, const float* targets, float* params, float* grads, float* adam_m,
                                   float* adam_v, float* bn_running, int32_t loss_kind, float* metrics, eims_stream_t stream,
                                   eims_stream_t side_stream) {
  if (!p || !p->blk) return fail(EIMS_ERR_STATE, "no step block set (eims_plan_set_step_block)");
  if (!targets && !p->peak_targets.peak_ptr) return fail(EIMS_ERR_ARG, "training needs target spectra");
  return enqueue_step(p, {targets, nullptr, nullptr, params, grads, adam_m, adam_v, bn_running, loss_kind, nullptr, metrics,
                          EIMS_BWD_ALL, (cudaStream_t)stream, (cudaStream_t)side_stream});
}

// The same step in two parts for a caller that runs its own optimiser between them (data-parallel training: the head
// bucket of the gradient exchange starts on a side stream when the head gradients are final, i.e. after part 1, and runs
// under the GraphConv backward of part 2).  No optimiser here.
int eims_train_step_built_indirect_part(eims_plan* p, const float* targets, float* params, float* grads, float* bn_running,
                                        int32_t loss_kind, float* metrics, int32_t part, eims_stream_t stream) {
  if (!p || !p->blk) return fail(EIMS_ERR_STATE, "no step block set (eims_plan_set_step_block)");
  if (part != 1 && part != 2) return fail(EIMS_ERR_ARG, "part must be 1 (forward, loss, head backward) or 2 (GraphConv backward)");
  if (part == 1 && !targets && !p->peak_targets.peak_ptr) return fail(EIMS_ERR_ARG, "training needs target spectra");
  return enqueue_step(p, {targets, nullptr, nullptr, params, grads, nullptr, nullptr, bn_running, loss_kind, nullptr, metrics,
                          part == 1 ? EIMS_BWD_HEAD : EIMS_BWD_GCN, (cudaStream_t)stream, nullptr});
}

int eims_infer_batch(eims_plan* p, const eims_dataset* ds, const int32_t* mol_ids, int32_t num_graphs,
                     const float* params, const float* bn_running, float* prob_out, eims_stream_t stream) {
  EIMS_TRY(eims_batch_build(p, ds, mol_ids, num_graphs, stream));
  EIMS_TRY(eims_forward(p, params, const_cast<float*>(bn_running), 0, nullptr, stream));
  cudaStream_t st = (cudaStream_t)stream;
  EarlyDimsScope early_scope(1);
  STAGE(ST_ELEMENTWISE, 1, launch_sigmoid(p->tab().dims, p->ws.logits, p->d.max_mz, prob_out ? prob_out : p->ws.prob, p->Bc,
                          (cudaStream_t)stream));
  return check_launch("eims_infer_batch");
}

int eims_plan_profile(eims_plan* p, int32_t enable) {
  if (!p) return fail(EIMS_ERR_ARG, "plan is NULL");
  p->prof = enable != 0;
  p->prof_used = 0;
  p->launches = 0;
  return 0;
}

int eims_plan_profile_read(eims_plan* p, float* stage_ms, int32_t* stage_launches, int32_t n_stages, int64_t* total_launches) {
  if (!p) return fail(EIMS_ERR_ARG, "plan is NULL");
  if (n_stages != ST_COUNT) return fail(EIMS_ERR_ARG, "n_stages must be %d", (int)ST_COUNT);
  if (cudaDeviceSynchronize() != cudaSuccess) return fail(EIMS_ERR_CUDA, "sync failed: %s", cudaGetErrorString(cudaGetLastError()));
  for (int k = 0; k < ST_COUNT; ++k) { if (stage_ms) stage_ms[k] = 0.f; if (stage_launches) stage_launches[k] = 0; }
  for (size_t k = 0; k < p->prof_used; ++k) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, p->prof_recs[k].a, p->prof_recs[k].b) != cudaSuccess)
      return fail(EIMS_ERR_CUDA, "cudaEventElapsedTime failed");
    if (stage_ms) stage_ms[p->prof_recs[k].stage] += ms;
    if (stage_launches) stage_launches[p->prof_recs[k].stage] += 1;
  }
  if (total_launches) *total_launches = p->launches;
  p->prof_used = 0;
  return 0;
}

int eims_plan_num_stages(void) { return ST_COUNT; }
const char* eims_plan_stage_name(int32_t k) { return (k >= 0 && k < ST_COUNT) ? kStageNames[k] : ""; }

int eims_plan_check(eims_plan* p, int32_t* num_nodes, int32_t* num_edges, eims_stream_t stream) {
  if (!p || !p->bound) return fail(EIMS_ERR_STATE, "plan not bound");
  int h[8];
  if (cudaMemcpyAsync(h, p->tab().dims, sizeof(h), cudaMemcpyDeviceToHost, (cudaStream_t)stream) != cudaSuccess ||
      cudaStreamSynchronize((cudaStream_t)stream) != cudaSuccess)
    return fail(EIMS_ERR_CUDA, "dims read-back failed: %s", cudaGetErrorString(cudaGetLastError()));
  if (num_nodes) *num_nodes = h[DIM_N];
  if (num_edges) *num_edges = h[DIM_E];
  if (h[DIM_OVERFLOW]) return fail(EIMS_ERR_CAPACITY, "batch exceeds plan capacity (max_nodes %d, max_edges %d) or a bond names an atom outside its molecule", p->Nc, p->Ec);
  if (h[DIM_ZERO_DEG] != 0 && h[DIM_ZERO_DEG] == h[5]) return fail(EIMS_ERR_ZERO_DEGREE, "There are 0-in-degree nodes in the graph (DGL GraphConv would raise)");
  return 0;
}


}  // extern "C"
#pragma GCC visibility pop

EIMS_TIMELINE_READER(plan)
