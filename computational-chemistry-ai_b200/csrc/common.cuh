// Shared device helpers for the EI-MS GCN kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/eims_b200.h"

#include <cmath>
#include <cstdlib>

namespace eims {

// dims[] slots written by K1 and read by every later kernel (sizes stay on the device so
// a captured step can be replayed for batches of any size up to the plan capacity).
enum { DIM_B = 0, DIM_N = 1, DIM_E = 2, DIM_ZERO_DEG = 3, DIM_OVERFLOW = 4, DIM_COUNT = 8 };

constexpr float kBnEps = 1e-5f;       // nn.BatchNorm1d default (GCN:317)
constexpr float kBnMomentum = 0.1f;   // nn.BatchNorm1d default
constexpr float kLnEps = 1e-5f;       // nn.LayerNorm default (GCN:343)
constexpr float kCosEps = 1e-8f;      // GCN:213-214

// Dropout sites: GCN layer l -> site l (GCN:362-363); head dropouts -> L, L+1 (GCN:345,349).
// torch's generator cannot be bit-matched, so the keep-mask is a counter-based stream of our
// own: two 32-bit hash words per 4 consecutive elements, keyed by a SplitMix64-derived 64-bit
// key of (seed, step, site), 16 random bits per element compared with p * 2^16.  It is a pure
// function of the element index, so the forward gather, the backward scatter and
// eims_dropout_mask all see the same mask without storing it.
struct DropCfg {
  uint32_t threshold;  // keep iff 16-bit word >= threshold ; threshold = round(p * 65536)
  float scale;         // 1/(1-p)
  uint64_t key;
  const uint64_t* key_dev;  // non-null: the key is read from the device-resident step block (captured CUDA graphs)
  __host__ __device__ bool active() const { return threshold != 0; }
};

__host__ __device__ __forceinline__ uint64_t mix64(uint64_t z) {
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  return z ^ (z >> 31);
}

static inline uint64_t drop_key(uint64_t seed, int step, int site) {
  return mix64(mix64(seed) ^ (((uint64_t)(uint32_t)step << 32) | (uint32_t)site));
}

static inline DropCfg make_drop(float p, uint64_t seed, int step, int site) {
  DropCfg d;
  double t = (double)p * 65536.0 + 0.5;
  d.threshold = p <= 0.f ? 0u : (t >= 65535.0 ? 65535u : (uint32_t)t);
  d.scale = p <= 0.f ? 1.f : 1.f / (1.f - p);
  d.key = drop_key(seed, step, site);
  d.key_dev = nullptr;
  return d;
}

// the kernel-side view: after the grid-dependency wait, take the key from the step block if there is one
__device__ __forceinline__ DropCfg resolve_drop(DropCfg d) {
  if (d.key_dev && d.threshold != 0u) d.key = __ldg(d.key_dev);
  return d;
}

// ---- device-resident per-step scalars ("step block")
// A captured CUDA graph freezes kernel parameters, so everything that changes from one optimiser step to
// the next - the molecule ids of the batch being built, the AdamW scalars (lr and beta1 follow the
// one-cycle schedule, GCN:386-391), the dropout keys, the data-parallel sequence number - lives in one
// small device struct that a 1-block kernel (parameters by value, so no host-buffer lifetime to manage)
// rewrites before every graph launch; the step's kernels read it instead of kernel parameters.
constexpr int kMaxDropSites = 24;
struct AdamK { float decay, one_minus_b1, b2, one_minus_b2, step_size, inv_bc2_sqrt, eps, grad_scale; };
// AdamW step scalars exactly as torch computes them (GCN:429): bias corrections with the CURRENT beta1
static inline AdamK make_adam_k(const eims_step* s) {
  const double b1 = s->beta1, b2 = s->beta2;
  const double bc1 = 1.0 - pow(b1, (double)s->step), bc2 = 1.0 - pow(b2, (double)s->step);
  AdamK k;
  k.decay = (float)(1.0 - (double)s->lr * (double)s->weight_decay);
  k.one_minus_b1 = (float)(1.0 - b1);
  k.b2 = (float)b2;
  k.one_minus_b2 = (float)(1.0 - b2);
  k.step_size = (float)((double)s->lr / bc1);
  k.inv_bc2_sqrt = (float)(1.0 / sqrt(bc2));
  k.eps = s->eps;
  k.grad_scale = s->grad_scale;
  return k;
}
struct StepBlock {
  const int32_t* ids;      // ids of the batch the indirect K1 builds
  AdamK adam;
  uint64_t drop_key[kMaxDropSites];
  uint32_t dp_seq;         // sequence number of the fused data-parallel exchange
  int32_t k1_seq;          // batch sequence number (tags the zero-degree flag)
};
constexpr int kStepPack = 16;   // blocks one upload launch can carry by value (kernel parameters are limited to 4 KB)
struct StepBlockPack { StepBlock b[kStepPack]; };
static_assert(sizeof(StepBlockPack) + 16 <= 4096, "step blocks no longer fit the kernel parameter space");

// 32-bit finaliser (two multiply / xor-shift rounds, the "lowbias32" constants of the hash-prospector
// search): ~8 integer instructions, against ~25 for a 64-bit SplitMix round on this machine - the forward
// SpMM hashes once per gathered float4 and is instruction-issue bound at BASELINE cfg 2 (ncu: IPC 2.1
// of 4, 38 % SM busy, 22 % memory).
__host__ __device__ __forceinline__ uint32_t mix32(uint32_t h) {
  h ^= h >> 16; h *= 0x21f0aaadu;
  h ^= h >> 15; h *= 0x735a2d97u;
  h ^= h >> 15;
  return h;
}

// keep-mask (scaled) for the 4 consecutive elements starting at flat index `elem` (elem % 4 == 0):
// two 32-bit words from the counter (elem / 4) and the 64-bit key, 16 random bits per element
__device__ __forceinline__ float4 drop_mask4(const DropCfg& d, uint64_t elem) {
  const uint32_t ctr = (uint32_t)(elem >> 2) ^ (uint32_t)(elem >> 34);
  const uint32_t lo = mix32(ctr * 0x9E3779B1u + (uint32_t)d.key);
  const uint32_t hi = mix32((lo ^ (uint32_t)(d.key >> 32)) * 0x85EBCA77u + ctr);
  float4 m;
  m.x = (lo & 0xffffu) >= d.threshold ? d.scale : 0.f;
  m.y = (lo >> 16) >= d.threshold ? d.scale : 0.f;
  m.z = (hi & 0xffffu) >= d.threshold ? d.scale : 0.f;
  m.w = (hi >> 16) >= d.threshold ? d.scale : 0.f;
  return m;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

// 3xTF32 operand split, the planes form (gemm_tma.cu): hi = rna_tf32(x), lo = rna_tf32(x - hi), both kept as fp32 bit
// patterns with the 13 low mantissa bits clear.  Round-to-nearest-away on the magnitude bits (+2^12, clear 13 bits):
// identical to cvt.rna.tf32.f32 for every finite input, and to the in-register split of gemm_tc.cu.
__device__ __forceinline__ void split_tf32_planes(float x, float& hi, float& lo) {
  hi = __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
  lo = __uint_as_float((__float_as_uint(x - hi) + 0x1000u) & 0xffffe000u);
}
__device__ __forceinline__ void split_tf32_planes4(float4 v, float4& h, float4& l) {
  split_tf32_planes(v.x, h.x, l.x); split_tf32_planes(v.y, h.y, l.y);
  split_tf32_planes(v.z, h.z, l.z); split_tf32_planes(v.w, h.w, l.w);
}

// Grid-wide "last block reduces" ticket.  Returns true in exactly one block (the last to
// arrive) after all earlier blocks' global writes are visible; resets the counter so the
// kernel can be relaunched / replayed from a CUDA graph.
__device__ __forceinline__ bool last_block_ticket(unsigned int* counter, unsigned int nblocks) {
  __shared__ bool is_last;
  // Release: the barrier orders every thread's earlier global writes / atomics before thread 0's
  // fence, and the fence is cumulative, so one fence per block (not one per thread) makes them
  // visible before the ticket is taken - the pattern cooperative-groups' grid sync uses.
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    unsigned int t = atomicAdd(counter, 1u);
    is_last = (t == nblocks - 1);
    if (is_last) *counter = 0u;
  }
  __syncthreads();
  if (is_last) __threadfence();  // acquire side, last block only
  return is_last;
}

// Programmatic dependent launch.  A step is a chain of ~35 short kernels (3-30 us each), so the
// launch latency and the prologue of kernel k+1 are overlapped with the tail of kernel k: every
// kernel is launched with the programmatic-stream-serialization attribute and starts with
// pdl_sync(): `griddepcontrol.wait` blocks until the preceding kernel has completed and its
// writes are visible (nothing - not even the device-side sizes in dims[] - is read before it),
// then `griddepcontrol.launch_dependents` lets the next kernel's blocks be scheduled as soon as
// this grid leaves room.
// -DEIMS_TIMELINE (tools/step_timeline.py; never in the product library): block 0 of every kernel
// stamps the global timer right after its grid-dependency wait, i.e. when the preceding kernel of
// the chain has completed, so consecutive stamps give the in-situ duration of every launch of a
// step with programmatic dependent launch left on.  Every translation unit keeps its own log
// (no relocatable device code needed) and exports a reader; the tool merges them by time.
#ifdef EIMS_TIMELINE
constexpr int kTimelineSlots = 8192;
static __device__ unsigned long long g_timeline[kTimelineSlots];
static __device__ unsigned int g_timeline_n;
#define EIMS_TIMELINE_READER(tu)                                                                                   \
  extern "C" __attribute__((visibility("default"))) int eims_debug_timeline_read_##tu(unsigned long long* out, int n) { \
    unsigned int used = 0;                                                                                         \
    if (cudaDeviceSynchronize() != cudaSuccess || cudaMemcpyFromSymbol(&used, eims::g_timeline_n, sizeof(used)) != cudaSuccess) return -2; \
    if ((int)used > n) used = (unsigned int)n;                                                                     \
    if (used && cudaMemcpyFromSymbol(out, eims::g_timeline, (size_t)used * sizeof(unsigned long long)) != cudaSuccess) return -2; \
    const unsigned int zero = 0;                                                                                   \
    if (cudaMemcpyToSymbol(eims::g_timeline_n, &zero, sizeof(zero)) != cudaSuccess) return -2;                      \
    return (int)used;                                                                                              \
  }
#else
#define EIMS_TIMELINE_READER(tu)
#endif

__device__ __forceinline__ void pdl_sync() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
#ifdef EIMS_TIMELINE
  if (threadIdx.x == 0 && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    const unsigned int i = atomicAdd(&g_timeline_n, 1u);
    if (i < kTimelineSlots) g_timeline[i] = t;
  }
#endif
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

// Batch sizes B / N / E of the current batch (dims[0..2], written by K1).  Every kernel needs them and used to read
// them first thing after the grid-dependency wait - a dependent L2 round trip at the head of every launch of a
// latency-bound step.  Under programmatic dependent launch a kernel that starts early overlaps only its immediate
// predecessor, whose own wait guarantees that everything before THAT has completed; so unless the predecessor is K1
// itself the sizes are already final when the kernel starts and can be loaded BEFORE the wait (`early` != 0).  The
// plan sets the flag for every launch of a step except the first one after the batch build (dims_early_ref()).
struct BatchDims { int B, N, E; };
__device__ __forceinline__ BatchDims pdl_sync_dims(const int* __restrict__ dims, int early) {
  int4 v = make_int4(0, 0, 0, 0);
  if (early) v = __ldcg(reinterpret_cast<const int4*>(dims));
  pdl_sync();
  if (!early) v = __ldcg(reinterpret_cast<const int4*>(dims));
  return BatchDims{v.x, v.y, v.z};
}
inline int& dims_early_ref() {
  static thread_local int v = 0;
  return v;
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// Training-mode BatchNorm1d statistics (GCN:361) fused into the kernel that produces z: the
// producer adds per-column sums of z and z^2 (fp64) into `acc`, and the last block to finish
// (ticket) turns them into mean / invstd / scale / shift, updates the running buffers
// (momentum 0.1, unbiased variance) and re-zeroes `acc` so the launch can be replayed.
// The fp64 column accumulators exist kBnReplicas times (block b adds into replica b % R, the
// finalizer sums them): hundreds of blocks finishing together would otherwise serialise their
// atomics on the handful of L2 slices that hold one 2*H*8-byte array.
constexpr int kBnReplicas = 8;
__device__ __forceinline__ double* bn_acc_slot(double* acc, int H, unsigned int block, int which, int col) {
  return acc + ((size_t)(block % kBnReplicas) * 2 + which) * H + col;
}
// sum of the replicas of one (statistic, column); re-zeroes them so the launch can be replayed
__device__ __forceinline__ double bn_acc_take(double* acc, int H, int which, int col) {
  double t = 0.0;
#pragma unroll
  for (int r = 0; r < kBnReplicas; ++r) {
    double* p = acc + ((size_t)r * 2 + which) * H + col;
    t += __ldcg(p);
    *p = 0.0;
  }
  return t;
}

struct BnFuse {
  double* acc;            // [kBnReplicas][2][H]; null = no fusion
  unsigned int* ticket;
  const float* gamma; const float* beta;
  float* running_mean; float* running_var;   // may be null
  float* mean; float* invstd; float* scale; float* shift;
  int H;
};

// executed by every thread of the finalizing block; n = rows the sums run over
__device__ __forceinline__ void bn_finalize(const BnFuse& f, int n_rows) {
  const double n = (double)n_rows;
  for (int c = threadIdx.x; c < f.H; c += blockDim.x) {
    const double s1 = bn_acc_take(f.acc, f.H, 0, c), s2 = bn_acc_take(f.acc, f.H, 1, c);
    if (n_rows <= 0) continue;
    const double mean = s1 / n;
    double var = s2 / n - mean * mean;
    if (var < 0.0) var = 0.0;
    const float mean_f = (float)mean;
    const float invstd = (float)(1.0 / sqrt(var + (double)kBnEps));
    f.mean[c] = mean_f;
    f.invstd[c] = invstd;
    const float sc = f.gamma[c] * invstd;
    f.scale[c] = sc;
    f.shift[c] = fmaf(-mean_f, sc, f.beta[c]);
    if (f.running_mean) {
      const float unbiased = (float)(n_rows > 1 ? var * n / (n - 1.0) : var);
      f.running_mean[c] = (1.f - kBnMomentum) * f.running_mean[c] + kBnMomentum * mean_f;
      f.running_var[c] = (1.f - kBnMomentum) * f.running_var[c] + kBnMomentum * unbiased;
    }
  }
}

}  // namespace eims
