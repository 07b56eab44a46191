// Dense-side kernels: BatchNorm statistics / backward, LayerNorm+ReLU+dropout, K7 fused
// sigmoid+MSE+cosine loss, column sums, K8 flat AdamW, and the CUDA-core fp32 GEMM that is the
// parity check path for the tcgen05 GEMM (gemm_tc.cu).
#include "common.cuh"
#include "launchers.h"

namespace eims {

// =========================================================================== fp32 SIMT GEMM
// C[M,N] = op(A) op(B); 64x64x16 tiles, 256 threads, 4x4 micro-tiles.  Check path only.
struct GemmArgs {
  const float* A; const float* B; float* C;
  int lda, ldb, ldc, a_mn, b_mn;
  int M, N, K;
  const int* m_dev; const int* k_dev;
  const float* row_scale; const float* bias;
  int relu, accumulate;
};

__global__ void __launch_bounds__(256) sgemm_simt_kernel(GemmArgs g) {
  pdl_sync();
  const int M = g.m_dev ? *g.m_dev : g.M;
  const int K = g.k_dev ? *g.k_dev : g.K;
  const int N = g.N;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  if (m0 >= M || n0 >= N) return;
  int kchunk = (K + gridDim.z - 1) / gridDim.z;
  kchunk = (kchunk + 15) & ~15;
  const int kbeg = blockIdx.z * kchunk, kend = min(K, kbeg + kchunk);
  if (kbeg >= kend && (g.accumulate || blockIdx.z > 0)) return;
  __shared__ float As[16][65];
  __shared__ float Bs[16][65];
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  float acc[4][4] = {};
  for (int k0 = kbeg; k0 < kend; k0 += 16) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int kk, mm;
      if (g.a_mn) { mm = t & 63; kk = (t >> 6) + 4 * i; } else { kk = t & 15; mm = (t >> 4) + 16 * i; }
      int m = m0 + mm, k = k0 + kk;
      float v = 0.f;
      if (m < M && k < kend) v = g.a_mn ? g.A[(int64_t)k * g.lda + m] : g.A[(int64_t)m * g.lda + k];
      As[kk][mm] = v;
      int nn;
      if (g.b_mn) { nn = t & 63; kk = (t >> 6) + 4 * i; } else { kk = t & 15; nn = (t >> 4) + 16 * i; }
      int n = n0 + nn;
      k = k0 + kk;
      v = 0.f;
      if (n < N && k < kend) v = g.b_mn ? g.B[(int64_t)k * g.ldb + n] : g.B[(int64_t)n * g.ldb + k];
      Bs[kk][nn] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[kk][ty * 4 + i]; b[i] = Bs[kk][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int m = m0 + ty * 4 + i;
    if (m >= M) continue;
    float rs = g.row_scale ? g.row_scale[m] : 1.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int n = n0 + tx * 4 + j;
      if (n >= N) continue;
      float v = acc[i][j] * rs + ((g.bias && blockIdx.z == 0) ? g.bias[n] : 0.f);
      if (g.relu) v = fmaxf(v, 0.f);
      if (g.accumulate) atomicAdd(g.C + (int64_t)m * g.ldc + n, v); else g.C[(int64_t)m * g.ldc + n] = v;
    }
  }
}

int launch_gemm_simt(const GemmProblem& q, cudaStream_t st) {
  const int M = q.M, N = q.N, K = q.K;
  if (M <= 0 || N <= 0 || K <= 0) return EIMS_ERR_ARG;
  // split-K-allowed store: plain store on this path
  const int accumulate = (q.accumulate == kGemmStoreSplit || q.accumulate == kGemmStoreSplitZeroed) ? 0 : q.accumulate;
  GemmArgs g{q.A, q.B, q.C, q.lda, q.ldb, q.ldc, q.a_mn, q.b_mn, M, N, K, q.m_dev, q.k_dev, q.row_scale, q.bias, q.relu, accumulate};
  int splits = 1;
  if (accumulate) {  // split-K for the weight gradients (K = atoms or graphs)
    int tiles = ((M + 63) / 64) * ((N + 63) / 64);
    splits = (148 * 4 + tiles - 1) / tiles;
    int maxs = (K + 63) / 64;
    if (splits > maxs) splits = maxs;
    if (splits < 1) splits = 1;
  }
  dim3 grid((N + 63) / 64, (M + 63) / 64, splits);
  launch_pdl(sgemm_simt_kernel, dim3(grid), dim3(256), 0, st, g);
  return 0;
}

// =========================================================================== BatchNorm column kernels
// Decomposition shared by the three kernels below: grid = (column slabs of 64, row groups),
// 256 threads = 16 float4 column lanes x 16 row lanes.  A thread strides over the rows of its
// row lane with its loads unrolled (memory-level parallelism is what these L2-resident passes
// need), the 16 row lanes are combined in shared memory, and each block issues one atomic per
// column and statistic - fp64 sums, so var = E[x^2]-mean^2 has no cancellation problem even for
// nearly constant columns.  The last block (ticket) finalises and re-zeroes the accumulators so
// the launch can be replayed.
constexpr int kSlab = 64, kRowLanes = 16;

// per_sm = blocks per SM in total: 4 (all resident at 64 registers) unless the kernel says otherwise
static inline dim3 bn_grid(int H, int max_nodes, int per_sm = 4) {
  const int slabs = (H + kSlab - 1) / kSlab;
  int rg = (148 * per_sm + slabs - 1) / slabs;
  const int need = (max_nodes + 4 * kRowLanes - 1) / (4 * kRowLanes);  // >= 4 rows per thread
  if (rg > need) rg = need;
  if (rg < 1) rg = 1;
  return dim3(slabs, rg);
}

// scratch: [16 floats: ticket counter] [kBnReplicas x 2H doubles: accumulators]
int64_t bn_scratch_floats(int H, int max_nodes) { (void)max_nodes; return 16 + 4 * (int64_t)H * kBnReplicas + 16; }

// combine the 16 row lanes of a block and add into acc[which*H + col] (fp64)
__device__ __forceinline__ void slab_reduce_atomic(const double (&a)[4], const double (&b)[4], int H, int c0, int cl,
                                                   int rl, double* acc) {
  __shared__ double red[kRowLanes][2][kSlab];
#pragma unroll
  for (int e = 0; e < 4; ++e) { red[rl][0][cl * 4 + e] = a[e]; red[rl][1][cl * 4 + e] = b[e]; }
  __syncthreads();
  if (threadIdx.x < 2 * kSlab) {
    const int which = threadIdx.x / kSlab, c = threadIdx.x % kSlab;
    double t = 0.0;
#pragma unroll
    for (int r = 0; r < kRowLanes; ++r) t += red[r][which][c];
    if (c0 + c < H) atomicAdd(bn_acc_slot(acc, H, blockIdx.y, which, c0 + c), t);
  }
}

__global__ void __launch_bounds__(256) bn_stats_kernel(const int* __restrict__ dims, const float* __restrict__ z, int H,
                                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                                       float* __restrict__ running_mean, float* __restrict__ running_var,
                                                       float* __restrict__ mean_out, float* __restrict__ invstd_out,
                                                       float* __restrict__ scale_out, float* __restrict__ shift_out,
                                                       float* __restrict__ scratch) {
  pdl_sync();
  const int N = dims[DIM_N];
  unsigned int* counter = reinterpret_cast<unsigned int*>(scratch);
  double* acc = reinterpret_cast<double*>(scratch + 16);
  const int cl = threadIdx.x & 15, rl = threadIdx.x >> 4;
  const int c0 = blockIdx.x * kSlab, c = c0 + cl * 4;
  double a[4] = {0.0, 0.0, 0.0, 0.0}, b[4] = {0.0, 0.0, 0.0, 0.0};
  if (c < H) {
    const int stride = gridDim.y * kRowLanes;
#pragma unroll 4
    for (int r = blockIdx.y * kRowLanes + rl; r < N; r += stride) {
      const float4 v = ldg4(z + (int64_t)r * H + c);
      const double x0 = v.x, x1 = v.y, x2 = v.z, x3 = v.w;
      a[0] += x0; a[1] += x1; a[2] += x2; a[3] += x3;
      b[0] = fma(x0, x0, b[0]); b[1] = fma(x1, x1, b[1]); b[2] = fma(x2, x2, b[2]); b[3] = fma(x3, x3, b[3]);
    }
  }
  slab_reduce_atomic(a, b, H, c0, cl, rl, acc);
  if (!last_block_ticket(counter, gridDim.x * gridDim.y)) return;
  BnFuse f{acc, counter, gamma, beta, running_mean, running_var, mean_out, invstd_out, scale_out, shift_out, H};
  bn_finalize(f, N);
}

int launch_bn_stats(const int* dims, const float* z, int H, const float* gamma, const float* beta, float* rmean,
                    float* rvar, float* mean, float* invstd, float* scale, float* shift, float* partials,
                    int max_nodes, cudaStream_t st) {
  if (H % 4 || H > 4096) return EIMS_ERR_ARG;
  launch_pdl(bn_stats_kernel, dim3(bn_grid(H, max_nodes)), dim3(256), 0, st, dims, z, H, gamma, beta, rmean, rvar, mean, invstd, scale,
                                                         shift, partials);
  return 0;
}

// eval-mode coefficients from the running buffers (GCN:442, model.eval()); mean / invstd (optional): the running
// mean and 1/sqrt(running_var + eps), which the eval-mode BatchNorm backward uses as its statistics
__global__ void bn_eval_coeffs_kernel(const float* __restrict__ gamma, const float* __restrict__ beta,
                                      const float* __restrict__ rmean, const float* __restrict__ rvar, int H,
                                      float* __restrict__ scale, float* __restrict__ shift, float* __restrict__ mean,
                                      float* __restrict__ invstd_out) {
  pdl_sync();
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < H; c += gridDim.x * blockDim.x) {
    float invstd = 1.f / sqrtf(rvar[c] + kBnEps);
    float sc = gamma[c] * invstd;
    scale[c] = sc;
    shift[c] = fmaf(-rmean[c], sc, beta[c]);
    if (mean) { mean[c] = rmean[c]; invstd_out[c] = invstd; }
  }
}
int launch_bn_eval_coeffs(const float* gamma, const float* beta, const float* rmean, const float* rvar, int H,
                          float* scale, float* shift, cudaStream_t st, float* mean, float* invstd) {
  if (!mean != !invstd) return EIMS_ERR_ARG;
  launch_pdl(bn_eval_coeffs_kernel, dim3((H + 255) / 256), dim3(256), 0, st, gamma, beta, rmean, rvar, H, scale, shift, mean, invstd);
  return 0;
}

// =========================================================================== BatchNorm backward
// dh source: either a materialised [N,H] buffer, or the readout backward computed on the fly
// from dG[B,pool_dim] (SumPooling/AvgPooling: broadcast; MaxPooling: first arg-max only).
struct DhSrc {
  const float* dh;       // [N,H] or null
  const float* dG;       // [B,pool_dim]
  const int* gid;        // [N]
  const int* gptr;       // [B+1]
  const int* argmax;     // [B,H]
  int pooling;
};

__device__ __forceinline__ float4 load_dh(const DhSrc& s, int i, int c, int H) {
  if (s.dh) return ldg4(s.dh + (int64_t)i * H + c);
  const int g = __ldg(s.gid + i);
  const int pd = s.pooling == EIMS_POOL_COMBINED ? 2 * H : H;
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (s.pooling != EIMS_POOL_MAX) {
    v = ldg4(s.dG + (int64_t)g * pd + c);
    if (s.pooling == EIMS_POOL_MEAN) {
      float n = (float)(__ldg(s.gptr + g + 1) - __ldg(s.gptr + g));
      v.x /= n; v.y /= n; v.z /= n; v.w /= n;
    }
  }
  if (s.pooling == EIMS_POOL_MAX || s.pooling == EIMS_POOL_COMBINED) {
    const int4 a = *reinterpret_cast<const int4*>(s.argmax + (int64_t)g * H + c);
    const float4 m = ldg4(s.dG + (int64_t)g * pd + (s.pooling == EIMS_POOL_COMBINED ? H : 0) + c);
    if (a.x == i) v.x += m.x;
    if (a.y == i) v.y += m.y;
    if (a.z == i) v.z += m.z;
    if (a.w == i) v.w += m.w;
  }
  return v;
}

// pass 1: column sums of dh and dh*xhat (fp64) -> dgamma, dbeta (into grads) and the two column means (means == NULL:
// not written - eval mode, where BatchNorm's output does not depend on the batch statistics and the apply pass takes
// zero means).
__global__ void __launch_bounds__(256, 4) bn_bwd_stats_kernel(const int* __restrict__ dims, const float* __restrict__ dh,
                                                           const float* __restrict__ z, int H,
                                                           const float* __restrict__ mean, const float* __restrict__ invstd,
                                                           float* __restrict__ dgamma, float* __restrict__ dbeta,
                                                           float* __restrict__ means /*[2][H]*/, float* __restrict__ scratch,
                                                           int early) {
  const int N = pdl_sync_dims(dims, early).N;
  unsigned int* counter = reinterpret_cast<unsigned int*>(scratch);
  double* acc = reinterpret_cast<double*>(scratch + 16);
  const int cl = threadIdx.x & 15, rl = threadIdx.x >> 4;
  const int c0 = blockIdx.x * kSlab, c = c0 + cl * 4;
  // per-thread partial sums in fp32 (a few rows each, no cancellation involved), fp64 from there on
  float af[4] = {0.f, 0.f, 0.f, 0.f}, bf[4] = {0.f, 0.f, 0.f, 0.f};
  if (c < H) {
    const float4 mu = ldg4(mean + c), is = ldg4(invstd + c);
    const int stride = gridDim.y * kRowLanes;
#pragma unroll 4
    for (int r = blockIdx.y * kRowLanes + rl; r < N; r += stride) {
      const float4 d = ldg4(dh + (int64_t)r * H + c);
      const float4 v = ldg4(z + (int64_t)r * H + c);
      af[0] += d.x; af[1] += d.y; af[2] += d.z; af[3] += d.w;
      bf[0] = fmaf(d.x, (v.x - mu.x) * is.x, bf[0]); bf[1] = fmaf(d.y, (v.y - mu.y) * is.y, bf[1]);
      bf[2] = fmaf(d.z, (v.z - mu.z) * is.z, bf[2]); bf[3] = fmaf(d.w, (v.w - mu.w) * is.w, bf[3]);
    }
  }
  double a[4], b[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) { a[e] = (double)af[e]; b[e] = (double)bf[e]; }
  slab_reduce_atomic(a, b, H, c0, cl, rl, acc);
  if (!last_block_ticket(counter, gridDim.x * gridDim.y)) return;
  for (int k = threadIdx.x; k < H; k += blockDim.x) {
    const double sa = bn_acc_take(acc, H, 0, k), sb = bn_acc_take(acc, H, 1, k);
    dbeta[k] += (float)sa;
    dgamma[k] += (float)sb;
    if (means) {
      means[k] = N > 0 ? (float)(sa / N) : 0.f;
      means[H + k] = N > 0 ? (float)(sb / N) : 0.f;
    }
  }
}

// The same statistics for the layer under the readout, without touching the nodes.  There
//   dh_i = dS_g (+ dMx_g at the arg-max node)        [sum; mean: dS_g / n_g; max: only the second term]
// so   sum_i dh_i       = sum_g ( n_g dS_g + dMx_g )
//      sum_i dh_i xhat_i = sum_g ( dS_g * Zsum_g + dMx_g * Zmax_g ) * invstd
// with Zsum_g = sum_{i in g} (z_i - mu) and Zmax_g = z_argmax - mu, which the readout kernel left in zstat:
// O(B*H) work instead of a pass over all N*H activations.  Thread = (column quad, graph lane).
__global__ void __launch_bounds__(256) bn_bwd_stats_top_kernel(const int* __restrict__ dims, const float* __restrict__ dG,
                                                               const float* __restrict__ zstat, const int* __restrict__ gptr,
                                                               int pooling, int H, const float* __restrict__ mean,
                                                               const float* __restrict__ invstd, float* __restrict__ dgamma,
                                                               float* __restrict__ dbeta, float* __restrict__ means,
                                                               float* __restrict__ scratch, int early) {
  const BatchDims bd = pdl_sync_dims(dims, early);
  const int B = bd.B, N = bd.N;
  unsigned int* counter = reinterpret_cast<unsigned int*>(scratch);
  double* acc = reinterpret_cast<double*>(scratch + 16);
  const int cl = threadIdx.x & 15, rl = threadIdx.x >> 4;
  const int c0 = blockIdx.x * kSlab, c = c0 + cl * 4;
  const int pd = pooling == EIMS_POOL_COMBINED ? 2 * H : H;
  double a[4] = {0.0, 0.0, 0.0, 0.0}, b[4] = {0.0, 0.0, 0.0, 0.0};
  if (c < H) {
    const float4 is = ldg4(invstd + c);
    for (int g = blockIdx.y * kRowLanes + rl; g < B; g += gridDim.y * kRowLanes) {
      const float n = (float)(__ldg(gptr + g + 1) - __ldg(gptr + g));
      if (pooling != EIMS_POOL_MAX) {
        float4 d = ldg4(dG + (int64_t)g * pd + c);
        const float4 zs = ldg4(zstat + (int64_t)g * 2 * H + c);
        if (pooling == EIMS_POOL_MEAN) { d.x /= n; d.y /= n; d.z /= n; d.w /= n; }  // every node of the graph gets dS / n
        a[0] += (double)d.x * n; a[1] += (double)d.y * n; a[2] += (double)d.z * n; a[3] += (double)d.w * n;
        b[0] += (double)d.x * (double)(zs.x * is.x); b[1] += (double)d.y * (double)(zs.y * is.y);
        b[2] += (double)d.z * (double)(zs.z * is.z); b[3] += (double)d.w * (double)(zs.w * is.w);
      }
      if ((pooling == EIMS_POOL_MAX || pooling == EIMS_POOL_COMBINED) && n > 0.f) {
        const float4 m = ldg4(dG + (int64_t)g * pd + (pooling == EIMS_POOL_COMBINED ? H : 0) + c);
        const float4 zm = ldg4(zstat + (int64_t)g * 2 * H + H + c);
        a[0] += (double)m.x; a[1] += (double)m.y; a[2] += (double)m.z; a[3] += (double)m.w;
        b[0] += (double)m.x * (double)(zm.x * is.x); b[1] += (double)m.y * (double)(zm.y * is.y);
        b[2] += (double)m.z * (double)(zm.z * is.z); b[3] += (double)m.w * (double)(zm.w * is.w);
      }
    }
  }
  slab_reduce_atomic(a, b, H, c0, cl, rl, acc);
  if (!last_block_ticket(counter, gridDim.x * gridDim.y)) return;
  for (int k = threadIdx.x; k < H; k += blockDim.x) {
    const double sa = bn_acc_take(acc, H, 0, k), sb = bn_acc_take(acc, H, 1, k);
    dbeta[k] += (float)sa;
    dgamma[k] += (float)sb;
    if (means) {
      means[k] = N > 0 ? (float)(sa / N) : 0.f;
      means[H + k] = N > 0 ? (float)(sb / N) : 0.f;
    }
  }
}

// zstat of an eval-mode forward, whose readout writes none: per graph, the column sums of z - mean (sum / mean
// pooling) and z - mean at the arg-max node (max pooling), mean = the running mean.  Thread = (graph, column quad).
__global__ void __launch_bounds__(256) bn_eval_zstat_kernel(const int* __restrict__ dims, const int* __restrict__ gptr,
                                                            const float* __restrict__ z, int H, const float* __restrict__ mean,
                                                            const int* __restrict__ argmax, int pooling,
                                                            float* __restrict__ zstat, int early) {
  const int B = pdl_sync_dims(dims, early).B;
  const int q4 = H >> 2;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < (int64_t)B * q4; t += (int64_t)gridDim.x * blockDim.x) {
    const int g = (int)(t / q4), c = (int)(t % q4) * 4;
    const int r0 = __ldg(gptr + g), r1 = __ldg(gptr + g + 1);
    const float4 mu = ldg4(mean + c);
    float* zo = zstat + (int64_t)g * 2 * H;
    if (pooling != EIMS_POOL_MAX) {
      float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int i = r0; i < r1; ++i) {
        const float4 v = ldg4(z + (int64_t)i * H + c);
        s.x += v.x - mu.x; s.y += v.y - mu.y; s.z += v.z - mu.z; s.w += v.w - mu.w;
      }
      st4(zo + c, s);
    }
    if ((pooling == EIMS_POOL_MAX || pooling == EIMS_POOL_COMBINED) && r1 > r0) {
      const int4 a = *reinterpret_cast<const int4*>(argmax + (int64_t)g * H + c);
      st4(zo + H + c, make_float4(__ldg(z + (int64_t)a.x * H + c) - mu.x, __ldg(z + (int64_t)a.y * H + c + 1) - mu.y,
                                  __ldg(z + (int64_t)a.z * H + c + 2) - mu.z, __ldg(z + (int64_t)a.w * H + c + 3) - mu.w));
    }
  }
}

int launch_bn_eval_zstat(const int* dims, const int* gptr, const float* z, int H, const float* mean, const int* argmax,
                         int pooling, float* zstat, int max_graphs, cudaStream_t st) {
  if (H % 4 || H > 4096) return EIMS_ERR_ARG;
  int64_t blocks = ((int64_t)max_graphs * (H / 4) + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  launch_pdl(bn_eval_zstat_kernel, dim3(blocks < 1 ? 1 : (int)blocks), dim3(256), 0, st, dims, gptr, z, H, mean,
             argmax, pooling, zstat, dims_early_ref());
  return 0;
}

int launch_bn_bwd_stats_top(const int* dims, const float* dG, const float* zstat, const int* gptr, int pooling, int H,
                            const float* mean, const float* invstd, float* dgamma, float* dbeta, float* means,
                            float* partials, int max_graphs, cudaStream_t st) {
  if (H % 4 || H > 4096) return EIMS_ERR_ARG;
  const int slabs = (H + kSlab - 1) / kSlab;
  // one graph per thread up to 37 row groups per slab (148 blocks at H = 256): the kernel is a chain of dependent
  // round trips (sizes -> operands -> shared-memory reduce -> atomics -> ticket -> finalize), so the four graphs a thread
  // used to walk one after the other were pure latency
  constexpr int kGraphsPerThread = 1;
  int rg = (max_graphs + kGraphsPerThread * kRowLanes - 1) / (kGraphsPerThread * kRowLanes);
  if (rg > 37) rg = 37;
  if (rg < 1) rg = 1;
  launch_pdl(bn_bwd_stats_top_kernel, dim3(slabs, rg), dim3(256), 0, st, dims, dG, zstat, gptr, pooling, H, mean, invstd, dgamma, dbeta,
             means, partials, dims_early_ref());
  return 0;
}

// pass 2: q = gamma*invstd*(dh - mean(dh) - xhat*mean(dh*xhat)) * [z>0] * c_i ;  dbias += colsum(dr)
// LAYER0: q is consumed on the spot by the first GraphConv's weight gradient dW0[f,k] += sum_i a0[i,f] * q[i,k]
// (F <= 8 rows); it is written (plain fp32) only when STORE_Q0, i.e. when the gradient w.r.t. the atom features is
// wanted (bn_bwd_apply_q0_kernel), and never by bn_bwd_apply_kernel<true>.
// DGRAD_ONLY (bn_apply_dgrad_kernel, the data-only eval backward of eims_attribute_peaks): q only - no bias gradient,
// no dW0, and the two column means are those of eval mode (zero), so they are not read.
constexpr int kMaxF0d = 8;

template <bool LAYER0, bool STORE_Q0, bool DGRAD_ONLY = false>
__device__ __forceinline__ void bn_bwd_apply_body(
    const int* __restrict__ dims, const DhSrc& src, const float* __restrict__ z, int H, const float* __restrict__ mean,
    const float* __restrict__ invstd, const float* __restrict__ gamma, const float* __restrict__ means,
    const float* __restrict__ norm, float* __restrict__ q, float* __restrict__ dbias, const float* __restrict__ a0,
    int F, float* __restrict__ dW0, int early, int64_t q_lo_off) {
  const int N = pdl_sync_dims(dims, early).N;
  __shared__ float red[kRowLanes][kSlab];
  const int cl = threadIdx.x & 15, rl = threadIdx.x >> 4;
  const int c0 = blockIdx.x * kSlab, c = c0 + cl * 4;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 w[LAYER0 ? kMaxF0d : 1];
#pragma unroll
  for (int f = 0; f < (LAYER0 ? kMaxF0d : 1); ++f) w[f] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (c < H) {
    const float4 mu = ldg4(mean + c), is = ldg4(invstd + c), ga = ldg4(gamma + c);
    const float4 m1 = DGRAD_ONLY ? make_float4(0.f, 0.f, 0.f, 0.f) : ldg4(means + c);
    const float4 m2 = DGRAD_ONLY ? make_float4(0.f, 0.f, 0.f, 0.f) : ldg4(means + H + c);
    const int stride = gridDim.y * kRowLanes;
#pragma unroll 4
    for (int r = blockIdx.y * kRowLanes + rl; r < N; r += stride) {
      const float4 d = load_dh(src, r, c, H);
      const float4 v = ldg4(z + (int64_t)r * H + c);
      const float ci = __ldg(norm + r);
      float4 o;
      o.x = v.x > 0.f ? ga.x * is.x * (d.x - m1.x - (v.x - mu.x) * is.x * m2.x) : 0.f;
      o.y = v.y > 0.f ? ga.y * is.y * (d.y - m1.y - (v.y - mu.y) * is.y * m2.y) : 0.f;
      o.z = v.z > 0.f ? ga.z * is.z * (d.z - m1.z - (v.z - mu.z) * is.z * m2.z) : 0.f;
      o.w = v.w > 0.f ? ga.w * is.w * (d.w - m1.w - (v.w - mu.w) * is.w * m2.w) : 0.f;
      if (!DGRAD_ONLY) { acc.x += o.x; acc.y += o.y; acc.z += o.z; acc.w += o.w; }
      o.x *= ci; o.y *= ci; o.z *= ci; o.w *= ci;
      if (LAYER0) {
#pragma unroll
        for (int f = 0; f < kMaxF0d; ++f)
          if (f < F) {
            const float a = __ldg(a0 + (int64_t)r * F + f);
            w[f].x = fmaf(a, o.x, w[f].x); w[f].y = fmaf(a, o.y, w[f].y);
            w[f].z = fmaf(a, o.z, w[f].z); w[f].w = fmaf(a, o.w, w[f].w);
          }
        if (STORE_Q0) st4(q + (int64_t)r * H + c, o);
      } else if (q_lo_off) {  // q as stacked tf32 hi / lo planes: the operand layout of gemm_tma.cu
        float4 hi4, lo4;
        split_tf32_planes4(o, hi4, lo4);
        st4(q + (int64_t)r * H + c, hi4);
        st4(q + q_lo_off + (int64_t)r * H + c, lo4);
      } else {
        st4(q + (int64_t)r * H + c, o);
      }
    }
    if (!LAYER0 && q_lo_off) {  // rows [N, next multiple of 32): zero in both planes (whole k-blocks of the weight gradient)
      for (int r = N + blockIdx.y * kRowLanes + rl; r < ((N + 31) & ~31); r += stride) {
        st4(q + (int64_t)r * H + c, make_float4(0.f, 0.f, 0.f, 0.f));
        st4(q + q_lo_off + (int64_t)r * H + c, make_float4(0.f, 0.f, 0.f, 0.f));
      }
    }
  }
  if (DGRAD_ONLY) return;
  red[rl][cl * 4 + 0] = acc.x; red[rl][cl * 4 + 1] = acc.y; red[rl][cl * 4 + 2] = acc.z; red[rl][cl * 4 + 3] = acc.w;
  __syncthreads();
  if (threadIdx.x < kSlab && c0 + threadIdx.x < H) {
    float t = 0.f;
#pragma unroll
    for (int r = 0; r < kRowLanes; ++r) t += red[r][threadIdx.x];
    atomicAdd(dbias + c0 + threadIdx.x, t);
  }
  if (LAYER0) {
    for (int f = 0; f < F; ++f) {
      __syncthreads();
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int k = 0; k < kMaxF0d; ++k)
        if (k == f) v = w[k];
      red[rl][cl * 4 + 0] = v.x; red[rl][cl * 4 + 1] = v.y; red[rl][cl * 4 + 2] = v.z; red[rl][cl * 4 + 3] = v.w;
      __syncthreads();
      if (threadIdx.x < kSlab && c0 + threadIdx.x < H) {
        float t = 0.f;
#pragma unroll
        for (int r = 0; r < kRowLanes; ++r) t += red[r][threadIdx.x];
        atomicAdd(dW0 + (int64_t)f * H + c0 + threadIdx.x, t);
      }
    }
  }
}

template <bool LAYER0>
__global__ void __launch_bounds__(256, LAYER0 ? 2 : 4) bn_bwd_apply_kernel(
    const int* __restrict__ dims, DhSrc src, const float* __restrict__ z, int H, const float* __restrict__ mean,
    const float* __restrict__ invstd, const float* __restrict__ gamma, const float* __restrict__ means,
    const float* __restrict__ norm, float* __restrict__ q, float* __restrict__ dbias, const float* __restrict__ a0,
    int F, float* __restrict__ dW0, int early, int64_t q_lo_off) {
  bn_bwd_apply_body<LAYER0, false>(dims, src, z, H, mean, invstd, gamma, means, norm, q, dbias, a0, F, dW0, early, q_lo_off);
}

// layer 0 when the gradient w.r.t. the atom features is wanted: the same pass, and q_0 = c * (dz_0 * relu') stored
__global__ void __launch_bounds__(256, 2) bn_bwd_apply_q0_kernel(
    const int* __restrict__ dims, DhSrc src, const float* __restrict__ z, int H, const float* __restrict__ mean,
    const float* __restrict__ invstd, const float* __restrict__ gamma, const float* __restrict__ means,
    const float* __restrict__ norm, float* __restrict__ q, float* __restrict__ dbias, const float* __restrict__ a0,
    int F, float* __restrict__ dW0, int early) {
  bn_bwd_apply_body<true, true>(dims, src, z, H, mean, invstd, gamma, means, norm, q, dbias, a0, F, dW0, early, 0);
}

// the data-only eval backward (eims_attribute_peaks): q = c * (gamma * invstd * dh) * [z > 0], nothing else
__global__ void __launch_bounds__(256, 4) bn_apply_dgrad_kernel(
    const int* __restrict__ dims, DhSrc src, const float* __restrict__ z, int H, const float* __restrict__ mean,
    const float* __restrict__ invstd, const float* __restrict__ gamma, const float* __restrict__ norm,
    float* __restrict__ q, int early, int64_t q_lo_off) {
  bn_bwd_apply_body<false, false, true>(dims, src, z, H, mean, invstd, gamma, nullptr, norm, q, nullptr, nullptr, 0, nullptr,
                                        early, q_lo_off);
}

int launch_bn_dgrad_apply(const int* dims, const float* dh, const float* dG, const int* gid, const int* gptr,
                          const int* argmax, int pooling, const float* z, int H, const float* mean, const float* invstd,
                          const float* gamma, const float* norm, float* q, int max_nodes, cudaStream_t st, int64_t q_lo_off) {
  if (H % 4 || H > 4096 || (q_lo_off & 3)) return EIMS_ERR_ARG;
  const DhSrc src{dh, dG, gid, gptr, argmax, pooling};
  launch_pdl(bn_apply_dgrad_kernel, bn_grid(H, max_nodes), dim3(256), 0, st, dims, src, z, H, mean, invstd, gamma, norm, q,
             dims_early_ref(), q_lo_off);
  return 0;
}

int launch_bn_bwd_stats(const int* dims, const float* dh, const float* z, int H, const float* mean, const float* invstd,
                        float* dgamma, float* dbeta, float* means, float* partials, int max_nodes, cudaStream_t st) {
  if (H % 4 || H > 4096) return EIMS_ERR_ARG;
  launch_pdl(bn_bwd_stats_kernel, bn_grid(H, max_nodes), dim3(256), 0, st, dims, dh, z, H, mean, invstd, dgamma, dbeta, means, partials,
             dims_early_ref());
  return 0;
}

int launch_bn_bwd_apply(const int* dims, const float* dh, const float* dG, const int* gid, const int* gptr,
                        const int* argmax, int pooling, const float* z, int H, const float* mean, const float* invstd,
                        const float* gamma, const float* norm, float* dbias, const float* means, float* q, int max_nodes,
                        cudaStream_t st, const float* a0, int F, float* dW0, int64_t q_lo_off, bool store_q0) {
  if (H % 4 || H > 4096 || (dW0 && (F < 1 || F > kMaxF0d)) || (q_lo_off & 3) || (dW0 && q_lo_off) || (store_q0 && !dW0))
    return EIMS_ERR_ARG;
  const DhSrc src{dh, dG, gid, gptr, argmax, pooling};
  const dim3 grid = bn_grid(H, max_nodes);
  // the layer-0 variant (104 registers: two resident blocks per SM) is launched as one wave: 12.7 us against 16.3
  constexpr int kL0BlocksPerSm = 2;
  if (store_q0)
    launch_pdl(bn_bwd_apply_q0_kernel, bn_grid(H, max_nodes, kL0BlocksPerSm), dim3(256), 0, st, dims, src, z, H, mean, invstd, gamma, means, norm, q, dbias, a0, F, dW0, dims_early_ref());
  else if (dW0)
    launch_pdl(bn_bwd_apply_kernel<true>, bn_grid(H, max_nodes, kL0BlocksPerSm), dim3(256), 0, st, dims, src, z, H, mean, invstd, gamma, means, norm, q, dbias, a0, F, dW0, dims_early_ref(), (int64_t)0);
  else
    launch_pdl(bn_bwd_apply_kernel<false>, grid, dim3(256), 0, st, dims, src, z, H, mean, invstd, gamma, means, norm, q, dbias, nullptr, 0, nullptr, dims_early_ref(), q_lo_off);
  return 0;
}

// =========================================================================== LayerNorm + ReLU + dropout
// Warp per row (GCN:343-345, 347-349).  Row kept in registers: NV float4 per lane, width <= 2048.
template <int NV>
__global__ void __launch_bounds__(256) ln_relu_drop_fwd_kernel(const int* __restrict__ dims, const float* __restrict__ u,
                                                               int W, const float* __restrict__ gamma,
                                                               const float* __restrict__ beta, DropCfg drop,
                                                               float* __restrict__ y, float* __restrict__ stats, int early) {
  const int B = pdl_sync_dims(dims, early).B;
  drop = resolve_drop(drop);
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int nv4 = W >> 2;
  for (int r = warp; r < B; r += nwarps) {
    float4 v[NV];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c4 = i * 32 + lane;
      v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c4 < nv4) {
        v[i] = ldg4(u + (int64_t)r * W + 4 * c4);
        s += v[i].x + v[i].y + v[i].z + v[i].w;
      }
    }
    const float mean = warp_sum(s) / (float)W;
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i)
      if (i * 32 + lane < nv4) {
        float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
        ss += a * a + b * b + c * c + d * d;
      }
    const float rstd = 1.f / sqrtf(warp_sum(ss) / (float)W + kLnEps);
    if (stats && lane == 0) { stats[2 * r] = mean; stats[2 * r + 1] = rstd; }
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c4 = i * 32 + lane;
      if (c4 < nv4) {
        const int c = 4 * c4;
        float4 g = ldg4(gamma + c), b = ldg4(beta + c), o;
        o.x = fmaxf(fmaf((v[i].x - mean) * rstd, g.x, b.x), 0.f);
        o.y = fmaxf(fmaf((v[i].y - mean) * rstd, g.y, b.y), 0.f);
        o.z = fmaxf(fmaf((v[i].z - mean) * rstd, g.z, b.z), 0.f);
        o.w = fmaxf(fmaf((v[i].w - mean) * rstd, g.w, b.w), 0.f);
        if (drop.active()) {
          float4 m = drop_mask4(drop, (uint64_t)r * W + c);
          o.x *= m.x; o.y *= m.y; o.z *= m.z; o.w *= m.w;
        }
        st4(y + (int64_t)r * W + c, o);
      }
    }
  }
}

static inline int ln_nv(int W) {
  int nv = (W + 127) / 128, p = 1;
  while (p < nv) p <<= 1;
  return p;
}

int launch_ln_fwd(const int* dims, const float* u, int W, const float* gamma, const float* beta, DropCfg drop, float* y,
                  float* stats, int max_graphs, cudaStream_t st) {
  if (W % 4 || W > 2048 || W < 4) return EIMS_ERR_ARG;
  int blocks = (max_graphs + 7) / 8;
  if (blocks < 1) blocks = 1;
  switch (ln_nv(W)) {
#define EIMS_LN_F(NV) case NV: launch_pdl(ln_relu_drop_fwd_kernel<NV>, dim3(blocks), dim3(256), 0, st, dims, u, W, gamma, beta, drop, y, stats, dims_early_ref()); break;
    EIMS_LN_F(1) EIMS_LN_F(2) EIMS_LN_F(4) EIMS_LN_F(8) EIMS_LN_F(16)
#undef EIMS_LN_F
    default: return EIMS_ERR_ARG;
  }
  return 0;
}

// backward: dy (grad w.r.t. the post-dropout output y) -> du (may alias dy); dgamma/dbeta += ;
// dbias (may be null) += column sums of du = bias gradient of the Linear that produced u.
template <int NV>
__global__ void __launch_bounds__(256) ln_relu_drop_bwd_kernel(const int* __restrict__ dims, const float* __restrict__ u,
                                                               const float* __restrict__ y, const float* dy, int W,
                                                               const float* __restrict__ gamma,
                                                               const float* __restrict__ stats, float drop_scale,
                                                               float* du, float* __restrict__ dgamma,
                                                               float* __restrict__ dbeta, float* __restrict__ dbias, int early) {
  extern __shared__ float smem[];  // [8 warps][3][W] : per-warp column partials of dgamma / dbeta / dbias
  const int B = pdl_sync_dims(dims, early).B;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int nv4 = W >> 2;
  float* sg = smem + (wib * 3 + 0) * W;
  float* sb = smem + (wib * 3 + 1) * W;
  float* sd = smem + (wib * 3 + 2) * W;
  for (int c = lane; c < W; c += 32) { sg[c] = 0.f; sb[c] = 0.f; sd[c] = 0.f; }
  __syncwarp();
  for (int r = warp; r < B; r += nwarps) {
    const float mean = stats[2 * r], rstd = stats[2 * r + 1];
    float4 xh[NV], g[NV];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c4 = i * 32 + lane;
      xh[i] = g[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c4 < nv4) {
        const int c = 4 * c4;
        float4 uu = ldg4(u + (int64_t)r * W + c), yy = ldg4(y + (int64_t)r * W + c);
        float4 d = *reinterpret_cast<const float4*>(dy + (int64_t)r * W + c);
        float4 ga = ldg4(gamma + c);
        float4 dt;
        dt.x = yy.x > 0.f ? d.x * drop_scale : 0.f; dt.y = yy.y > 0.f ? d.y * drop_scale : 0.f;
        dt.z = yy.z > 0.f ? d.z * drop_scale : 0.f; dt.w = yy.w > 0.f ? d.w * drop_scale : 0.f;
        xh[i].x = (uu.x - mean) * rstd; xh[i].y = (uu.y - mean) * rstd;
        xh[i].z = (uu.z - mean) * rstd; xh[i].w = (uu.w - mean) * rstd;
        float4 a = *reinterpret_cast<float4*>(sg + c), b = *reinterpret_cast<float4*>(sb + c);
        a.x = fmaf(dt.x, xh[i].x, a.x); a.y = fmaf(dt.y, xh[i].y, a.y);
        a.z = fmaf(dt.z, xh[i].z, a.z); a.w = fmaf(dt.w, xh[i].w, a.w);
        b.x += dt.x; b.y += dt.y; b.z += dt.z; b.w += dt.w;
        *reinterpret_cast<float4*>(sg + c) = a;
        *reinterpret_cast<float4*>(sb + c) = b;
        g[i].x = dt.x * ga.x; g[i].y = dt.y * ga.y; g[i].z = dt.z * ga.z; g[i].w = dt.w * ga.w;
        s1 += g[i].x + g[i].y + g[i].z + g[i].w;
        s2 += g[i].x * xh[i].x + g[i].y * xh[i].y + g[i].z * xh[i].z + g[i].w * xh[i].w;
      }
    }
    const float m1 = warp_sum(s1) / (float)W, m2 = warp_sum(s2) / (float)W;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c4 = i * 32 + lane;
      if (c4 < nv4) {
        float4 o;
        o.x = rstd * (g[i].x - m1 - xh[i].x * m2); o.y = rstd * (g[i].y - m1 - xh[i].y * m2);
        o.z = rstd * (g[i].z - m1 - xh[i].z * m2); o.w = rstd * (g[i].w - m1 - xh[i].w * m2);
        st4(du + (int64_t)r * W + 4 * c4, o);
        float4 d4 = *reinterpret_cast<float4*>(sd + 4 * c4);
        d4.x += o.x; d4.y += o.y; d4.z += o.z; d4.w += o.w;
        *reinterpret_cast<float4*>(sd + 4 * c4) = d4;
      }
    }
  }
  __syncthreads();
  const int nw = blockDim.x >> 5;
  for (int c = threadIdx.x; c < W; c += blockDim.x) {
    float a = 0.f, b = 0.f, d = 0.f;
    for (int w = 0; w < nw; ++w) { a += smem[(w * 3) * W + c]; b += smem[(w * 3 + 1) * W + c]; d += smem[(w * 3 + 2) * W + c]; }
    atomicAdd(dgamma + c, a);
    atomicAdd(dbeta + c, b);
    if (dbias) atomicAdd(dbias + c, d);
  }
}

int launch_ln_bwd(const int* dims, const float* u, const float* y, const float* dy, int W, const float* gamma,
                  const float* stats, float drop_scale, float* du, float* dgamma, float* dbeta, float* dbias,
                  int max_graphs, cudaStream_t st) {
  if (W % 4 || W > 2048 || W < 4) return EIMS_ERR_ARG;
  constexpr int kRowsPerBlock = 8;  // (8 warps): one row per warp measured best (cfg 2: 9.7 us for the two launches, 11.9 with two rows)
  int blocks = (max_graphs + kRowsPerBlock - 1) / kRowsPerBlock;
  if (blocks < 1) blocks = 1;
  if (blocks > 148) blocks = 148;
  size_t smem = (size_t)8 * 3 * W * sizeof(float);
  switch (ln_nv(W)) {
#define EIMS_LN_B(NV)                                                                                              \
  case NV:                                                                                                         \
    if (smem > 48 * 1024)                                                                                          \
      cudaFuncSetAttribute(ln_relu_drop_bwd_kernel<NV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);   \
    launch_pdl(ln_relu_drop_bwd_kernel<NV>, dim3(blocks), dim3(256), smem, st, dims, u, y, dy, W, gamma, stats, drop_scale, du, dgamma, dbeta, dbias, dims_early_ref()); \
    break;
    EIMS_LN_B(1) EIMS_LN_B(2) EIMS_LN_B(4) EIMS_LN_B(8) EIMS_LN_B(16)
#undef EIMS_LN_B
    default: return EIMS_ERR_ARG;
  }
  return 0;
}

// data-only backward of eval mode (eims_attribute_peaks): du only, no dgamma / dbeta / bias gradient (and so no shared
// partials and no atomics); no dropout.  du may alias dy.  Warp per row, the arithmetic of ln_relu_drop_bwd_kernel.
template <int NV>
__global__ void __launch_bounds__(256) ln_relu_dgrad_kernel(const int* __restrict__ dims, const float* __restrict__ u,
                                                            const float* __restrict__ y, const float* dy, int W,
                                                            const float* __restrict__ gamma, const float* __restrict__ stats,
                                                            float* du, int early) {
  const int B = pdl_sync_dims(dims, early).B;
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int nv4 = W >> 2;
  for (int r = warp; r < B; r += nwarps) {
    const float mean = stats[2 * r], rstd = stats[2 * r + 1];
    float4 xh[NV], g[NV];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c4 = i * 32 + lane;
      xh[i] = g[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c4 < nv4) {
        const int c = 4 * c4;
        const float4 uu = ldg4(u + (int64_t)r * W + c), yy = ldg4(y + (int64_t)r * W + c), ga = ldg4(gamma + c);
        const float4 d = *reinterpret_cast<const float4*>(dy + (int64_t)r * W + c);
        xh[i].x = (uu.x - mean) * rstd; xh[i].y = (uu.y - mean) * rstd;
        xh[i].z = (uu.z - mean) * rstd; xh[i].w = (uu.w - mean) * rstd;
        g[i].x = yy.x > 0.f ? d.x * ga.x : 0.f; g[i].y = yy.y > 0.f ? d.y * ga.y : 0.f;
        g[i].z = yy.z > 0.f ? d.z * ga.z : 0.f; g[i].w = yy.w > 0.f ? d.w * ga.w : 0.f;
        s1 += g[i].x + g[i].y + g[i].z + g[i].w;
        s2 += g[i].x * xh[i].x + g[i].y * xh[i].y + g[i].z * xh[i].z + g[i].w * xh[i].w;
      }
    }
    const float m1 = warp_sum(s1) / (float)W, m2 = warp_sum(s2) / (float)W;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c4 = i * 32 + lane;
      if (c4 < nv4) {
        float4 o;
        o.x = rstd * (g[i].x - m1 - xh[i].x * m2); o.y = rstd * (g[i].y - m1 - xh[i].y * m2);
        o.z = rstd * (g[i].z - m1 - xh[i].z * m2); o.w = rstd * (g[i].w - m1 - xh[i].w * m2);
        st4(du + (int64_t)r * W + 4 * c4, o);
      }
    }
  }
}

int launch_ln_dgrad(const int* dims, const float* u, const float* y, const float* dy, int W, const float* gamma,
                    const float* stats, float* du, int max_graphs, cudaStream_t st) {
  if (W % 4 || W > 2048 || W < 4) return EIMS_ERR_ARG;
  int blocks = (max_graphs + 7) / 8;  // 8 warps, one row each
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  switch (ln_nv(W)) {
#define EIMS_LN_D(NV) case NV: launch_pdl(ln_relu_dgrad_kernel<NV>, dim3(blocks), dim3(256), 0, st, dims, u, y, dy, W, gamma, stats, du, dims_early_ref()); break;
    EIMS_LN_D(1) EIMS_LN_D(2) EIMS_LN_D(4) EIMS_LN_D(8) EIMS_LN_D(16)
#undef EIMS_LN_D
    default: return EIMS_ERR_ARG;
  }
  return 0;
}

// =========================================================================== peaks of eims_attribute_peaks
// The head's first data gradient for dprob = one-hot(m_r) per row: dlogits is p (1 - p) at m_r and zero elsewhere, so
// dy2[r, :] = p (1 - p) W3[m_r, :] with p = sigmoid(logits[r, m_r]) - a gather instead of the [B, M] x [M, H] GEMM.
// Warp per row.
__global__ void __launch_bounds__(256) peak_head_dgrad_kernel(const int* __restrict__ dims, const float* __restrict__ logits,
                                                              int M, const int* __restrict__ bins, const float* __restrict__ W3,
                                                              int H, float* __restrict__ dy2, int early) {
  const int B = pdl_sync_dims(dims, early).B;
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int r = warp; r < B; r += nwarps) {
    const int m = __ldg(bins + r);
    const float p = 1.f / (1.f + expf(-__ldg(logits + (int64_t)r * M + m)));
    const float s = p * (1.f - p);
    for (int c = 4 * lane; c < H; c += 128) {
      float4 w = ldg4(W3 + (int64_t)m * H + c);
      w.x *= s; w.y *= s; w.z *= s; w.w *= s;
      st4(dy2 + (int64_t)r * H + c, w);
    }
  }
}

// idx / val: the top-k table [rows, k] of the predicted spectra.  Graph r takes entry r mod k (the host layer puts every
// molecule k times in a row, so the k replicas of a molecule take its k peaks).
__global__ void peak_select_kernel(const int* __restrict__ dims, const int* __restrict__ idx, const float* __restrict__ val,
                                   int k, int* __restrict__ bins, float* __restrict__ prob, int early) {
  const int B = pdl_sync_dims(dims, early).B;
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < B; r += gridDim.x * blockDim.x) {
    const int64_t e = (int64_t)r * k + r % k;
    bins[r] = __ldg(idx + e);
    prob[r] = __ldg(val + e);
  }
}

// prob[r] = sigmoid(logits[r, bins[r]]) (the arithmetic of sigmoid_kernel)
__global__ void peak_prob_kernel(const int* __restrict__ dims, const float* __restrict__ logits, int M,
                                 const int* __restrict__ bins, float* __restrict__ prob, int early) {
  const int B = pdl_sync_dims(dims, early).B;
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < B; r += gridDim.x * blockDim.x)
    prob[r] = 1.f / (1.f + expf(-__ldg(logits + (int64_t)r * M + __ldg(bins + r))));
}

static inline int row_blocks(int rows, int per_block) {
  int b = (rows + per_block - 1) / per_block;
  if (b > 148 * 8) b = 148 * 8;
  return b < 1 ? 1 : b;
}

int launch_peak_head_dgrad(const int* dims, const float* logits, int M, const int* bins, const float* W3, int H, float* dy2,
                           int max_graphs, cudaStream_t st) {
  if (H % 4) return EIMS_ERR_ARG;
  launch_pdl(peak_head_dgrad_kernel, dim3(row_blocks(max_graphs, 8)), dim3(256), 0, st, dims, logits, M, bins, W3, H, dy2,
             dims_early_ref());
  return 0;
}

int launch_peak_select(const int* dims, const int* idx, const float* val, int k, int* bins, float* prob, int max_graphs,
                       cudaStream_t st) {
  launch_pdl(peak_select_kernel, dim3(row_blocks(max_graphs, 256)), dim3(256), 0, st, dims, idx, val, k, bins, prob,
             dims_early_ref());
  return 0;
}

int launch_peak_prob(const int* dims, const float* logits, int M, const int* bins, float* prob, int max_graphs,
                     cudaStream_t st) {
  launch_pdl(peak_prob_kernel, dim3(row_blocks(max_graphs, 256)), dim3(256), 0, st, dims, logits, M, bins, prob,
             dims_early_ref());
  return 0;
}

// =========================================================================== K7 loss
// Block (128 threads) per graph: prob = sigmoid(logits); MSE and cosine terms; dlogits.
constexpr int kLossMaxV4 = 8;  // max_mz <= 4096

__device__ __forceinline__ float block_sum_128(float v, float* sh) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  return sh[0] + sh[1] + sh[2] + sh[3];
}

// metrics += {mean loss, mean cos, 1}; [4],[5] = this step's values.  One block, fixed summation
// order (deterministic).  This is the per-step `loss.item()` / `cos_sim.mean().item()` of
// GCN:436-437 kept on the device.
__device__ __forceinline__ void metrics_reduce(int B, const float* row_loss, const float* row_cos, int M, float* metrics) {
  __shared__ double s1[256], s2[256];
  double a = 0.0, b = 0.0;
  for (int i = threadIdx.x; i < B; i += blockDim.x) { a += (double)__ldcg(row_loss + i); b += (double)__ldcg(row_cos + i); }
  if (threadIdx.x < 256) { s1[threadIdx.x] = a; s2[threadIdx.x] = b; }
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o && threadIdx.x + o < blockDim.x) { s1[threadIdx.x] += s1[threadIdx.x + o]; s2[threadIdx.x] += s2[threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0 && B > 0) {
    const float loss = (float)(s1[0] / ((double)B * (double)M));
    const float cosm = (float)(s2[0] / (double)B);
    metrics[0] += loss; metrics[1] += cosm; metrics[2] += 1.f;
    metrics[4] = loss; metrics[5] = cosm;  // last step's values
    if (!isfinite(loss)) metrics[6] += 1.f;  // NaN / Inf guard: steps whose loss was not finite (read once per epoch)
  }
}

// ---- peak list -> spectrum (CuPySpectrumProcessor.peaks_to_spectrum_batch, GCN:166-205)
// One block (128 threads) bins one spectrum into `bins` (shared, M floats): zero, scatter-max,
// row maximum.  Non-negative floats order like their bit patterns, so the max-merge is an integer
// atomicMax in shared memory; intensities <= 0 / NaN never replace the initial 0 (the reference's
// max(spectra[i, k], intensity) keeps its first argument unless the second is greater).
// Returns the divisor: the row maximum, or 1 for an all-zero row (GCN:200-201).
struct PeakSrc { const int64_t* ptr; const void* mz; const float* inten; int is_f64; };

__device__ __forceinline__ float bin_peaks_row(const PeakSrc& pk, int64_t row, int M, float* bins, float* sh) {
  for (int c = threadIdx.x; c < M; c += 128) bins[c] = 0.f;
  __syncthreads();
  const int64_t k0 = pk.ptr[row], k1 = pk.ptr[row + 1];
  for (int64_t k = k0 + threadIdx.x; k < k1; k += 128) {
    // np.round / cp.round: to nearest, ties to even, in the precision the m/z is stored in
    const double r = pk.is_f64 ? rint(reinterpret_cast<const double*>(pk.mz)[k])
                               : (double)rintf(reinterpret_cast<const float*>(pk.mz)[k]);
    const float v = pk.inten[k];
    if (r >= 0.0 && r < (double)M && v > 0.f) atomicMax(reinterpret_cast<int*>(bins) + (int)r, __float_as_int(v));
  }
  __syncthreads();
  float mx = 0.f;
  for (int c = threadIdx.x; c < M; c += 128) mx = fmaxf(mx, bins[c]);
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = mx;
  __syncthreads();
  mx = fmaxf(fmaxf(sh[0], sh[1]), fmaxf(sh[2], sh[3]));
  __syncthreads();
  return mx > 0.f ? mx : 1.f;
}

__global__ void __launch_bounds__(128) peaks_to_spectrum_kernel(PeakSrc pk, const int* __restrict__ rows, int num_rows,
                                                                int M, float* __restrict__ out) {
  pdl_sync();
  __shared__ float bins[4 * 128 * 8];
  __shared__ float sh[4];
  for (int b = blockIdx.x; b < num_rows; b += gridDim.x) {
    const float mx = bin_peaks_row(pk, rows ? (int64_t)rows[b] : (int64_t)b, M, bins, sh);
    for (int c = threadIdx.x; c < M; c += 128) out[(int64_t)b * M + c] = __fdiv_rn(bins[c], mx);
    __syncthreads();
  }
}

int launch_peaks_to_spectrum(const eims_peaks* pk, const int* rows, int num_rows, int M, float* out, cudaStream_t st) {
  if (!pk || !pk->peak_ptr || !pk->mz || !pk->intensity || !out || M < 1 || M > 4096 || num_rows < 0) return EIMS_ERR_ARG;
  if (num_rows == 0) return 0;
  PeakSrc src{pk->peak_ptr, pk->mz, pk->intensity, pk->mz_is_f64};
  const int blocks = num_rows < 148 * 16 ? num_rows : 148 * 16;
  launch_pdl(peaks_to_spectrum_kernel, dim3(blocks), dim3(128), 0, st, src, rows, num_rows, M, out);
  return 0;
}

template <bool PEAKS>
__global__ void __launch_bounds__(128) loss_kernel(const int* __restrict__ dims, const float* __restrict__ logits,
                                                   const float* __restrict__ targets, const int* __restrict__ target_rows,
                                                   int M, int loss_kind, float* __restrict__ prob,
                                                   float* __restrict__ dlogits, float* __restrict__ row_loss,
                                                   float* __restrict__ row_cos, float* __restrict__ metrics,
                                                   unsigned int* __restrict__ ticket, PeakSrc pk, int early) {
  __shared__ float sh[4];
  __shared__ __align__(16) float bins[PEAKS ? 4 * 128 * kLossMaxV4 : 4];  // PEAKS: the target row is binned here
  const int B = pdl_sync_dims(dims, early).B;
  const int nv4 = M >> 2;
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    const int64_t trow = target_rows ? (int64_t)target_rows[b] : (int64_t)b;
    const float* t = targets + trow * M;
    float tmax = 1.f;
    if (PEAKS) tmax = bin_peaks_row(pk, trow, M, bins, sh);
    float4 p[kLossMaxV4], tt[kLossMaxV4];
    float se = 0.f, pp = 0.f, tq = 0.f, pt = 0.f;
#pragma unroll
    for (int i = 0; i < kLossMaxV4; ++i) {
      const int c4 = i * 128 + threadIdx.x;
      if (c4 < nv4) {
        float4 u = ldg4(logits + (int64_t)b * M + 4 * c4);
        if (PEAKS) {
          const float4 raw = *reinterpret_cast<const float4*>(bins + 4 * c4);
          tt[i] = make_float4(__fdiv_rn(raw.x, tmax), __fdiv_rn(raw.y, tmax), __fdiv_rn(raw.z, tmax), __fdiv_rn(raw.w, tmax));
        } else {
          tt[i] = ldg4(t + 4 * c4);
        }
        p[i].x = 1.f / (1.f + expf(-u.x)); p[i].y = 1.f / (1.f + expf(-u.y));
        p[i].z = 1.f / (1.f + expf(-u.z)); p[i].w = 1.f / (1.f + expf(-u.w));
        float dx = p[i].x - tt[i].x, dy = p[i].y - tt[i].y, dz = p[i].z - tt[i].z, dw = p[i].w - tt[i].w;
        se += dx * dx + dy * dy + dz * dz + dw * dw;
        pp += p[i].x * p[i].x + p[i].y * p[i].y + p[i].z * p[i].z + p[i].w * p[i].w;
        tq += tt[i].x * tt[i].x + tt[i].y * tt[i].y + tt[i].z * tt[i].z + tt[i].w * tt[i].w;
        pt += p[i].x * tt[i].x + p[i].y * tt[i].y + p[i].z * tt[i].z + p[i].w * tt[i].w;
        if (prob) st4(prob + (int64_t)b * M + 4 * c4, p[i]);
      }
    }
    se = block_sum_128(se, sh);
    pp = block_sum_128(pp, sh);
    tq = block_sum_128(tq, sh);
    pt = block_sum_128(pt, sh);
    const float np = sqrtf(pp) + kCosEps, nt = sqrtf(tq) + kCosEps;
    const float cosv = pt / (np * nt);
    if (threadIdx.x == 0) { row_loss[b] = se; row_cos[b] = cosv; }
    if (dlogits) {
      const float k_mse = 2.f / ((float)B * (float)M);
      // d(1-mean cos)/dp = -(1/B) * ( t/(nt*np) - cos * p / (||p|| * np) )
      const float ka = -1.f / ((float)B * nt * np);
      const float kb = cosv / ((float)B * fmaxf(sqrtf(pp), 1e-30f) * np);
#pragma unroll
      for (int i = 0; i < kLossMaxV4; ++i) {
        const int c4 = i * 128 + threadIdx.x;
        if (c4 < nv4) {
          float4 d;
          if (loss_kind == EIMS_LOSS_MSE) {
            d.x = k_mse * (p[i].x - tt[i].x); d.y = k_mse * (p[i].y - tt[i].y);
            d.z = k_mse * (p[i].z - tt[i].z); d.w = k_mse * (p[i].w - tt[i].w);
          } else {
            d.x = ka * tt[i].x + kb * p[i].x; d.y = ka * tt[i].y + kb * p[i].y;
            d.z = ka * tt[i].z + kb * p[i].z; d.w = ka * tt[i].w + kb * p[i].w;
          }
          d.x *= p[i].x * (1.f - p[i].x); d.y *= p[i].y * (1.f - p[i].y);
          d.z *= p[i].z * (1.f - p[i].z); d.w *= p[i].w * (1.f - p[i].w);
          st4(dlogits + (int64_t)b * M + 4 * c4, d);
        }
      }
    }
  }
  // the last block to finish folds the row terms into the running metrics (no extra launch)
  if (metrics && last_block_ticket(ticket, gridDim.x)) metrics_reduce(B, row_loss, row_cos, M, metrics);
}

int launch_loss(const int* dims, const float* logits, const float* targets, const int* target_rows, int M,
                int loss_kind, float* prob, float* dlogits, float* row_loss, float* row_cos, int max_graphs,
                cudaStream_t st, float* metrics, unsigned int* ticket, const eims_peaks* peaks) {
  if (M % 4 || M > 4 * 128 * kLossMaxV4 || (metrics && !ticket)) return EIMS_ERR_ARG;
  if (!targets && !(peaks && peaks->peak_ptr && peaks->mz && peaks->intensity)) return EIMS_ERR_ARG;
  PeakSrc src{nullptr, nullptr, nullptr, 0};
  if (!targets) src = PeakSrc{peaks->peak_ptr, peaks->mz, peaks->intensity, peaks->mz_is_f64};
  int blocks = max_graphs < 1 ? 1 : max_graphs;
  if (src.ptr)
    launch_pdl(loss_kernel<true>, dim3(blocks), dim3(128), 0, st, dims, logits, targets, target_rows, M, loss_kind, prob, dlogits,
               row_loss, row_cos, metrics, ticket, src, dims_early_ref());
  else
    launch_pdl(loss_kernel<false>, dim3(blocks), dim3(128), 0, st, dims, logits, targets, target_rows, M, loss_kind, prob, dlogits,
               row_loss, row_cos, metrics, ticket, src, dims_early_ref());
  return 0;
}

// ---- top-k peaks of predicted spectra (the report of `--mode predict`, GCN:610-613)
// Block (128 threads) per spectrum, k selection rounds: every thread keeps its M/128 bins in
// registers, a round is a block arg-max over the bins not taken yet.  Order: value descending,
// ties to the HIGHER bin - what np.argsort(spectrum, kind="stable")[-k:][::-1] gives (the
// reference's default-kind argsort leaves the order of exact ties unspecified).
constexpr int kTopkMaxPerThread = 32;  // max_mz <= 4096

__global__ void __launch_bounds__(128) topk_peaks_kernel(const float* __restrict__ spectra, int num_rows, int M, int k,
                                                         int* __restrict__ idx_out, float* __restrict__ val_out) {
  pdl_sync();
  __shared__ float sv[4];
  __shared__ int si[4];
  const float ninf = -__int_as_float(0x7f800000);
  for (int b = blockIdx.x; b < num_rows; b += gridDim.x) {
    float v[kTopkMaxPerThread];
    unsigned int taken = 0u;  // bit i: bin i*128+tid is out of the race (selected already, or past M)
#pragma unroll
    for (int i = 0; i < kTopkMaxPerThread; ++i) {
      const int c = i * 128 + threadIdx.x;
      v[i] = c < M ? __ldg(spectra + (int64_t)b * M + c) : ninf;
      if (!(v[i] == v[i])) v[i] = ninf;  // NaN ranks last
      if (c >= M) taken |= 1u << i;
    }
    for (int r = 0; r < k; ++r) {
      float bv = ninf;
      int bi = -1;
#pragma unroll
      for (int i = 0; i < kTopkMaxPerThread; ++i)
        if (!((taken >> i) & 1u) && (bi < 0 || v[i] >= bv)) { bv = v[i]; bi = i * 128 + threadIdx.x; }  // higher bin wins ties
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi > bi))) { bv = ov; bi = oi; }
      }
      __syncthreads();
      if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = bv; si[threadIdx.x >> 5] = bi; }
      __syncthreads();
      bv = sv[0]; bi = si[0];
#pragma unroll
      for (int w = 1; w < 4; ++w)
        if (si[w] >= 0 && (bi < 0 || sv[w] > bv || (sv[w] == bv && si[w] > bi))) { bv = sv[w]; bi = si[w]; }
      if (threadIdx.x == 0) {
        idx_out[(int64_t)b * k + r] = bi;
        if (val_out) val_out[(int64_t)b * k + r] = bv;
      }
      if (bi >= 0 && (bi & 127) == (int)threadIdx.x) taken |= 1u << (bi >> 7);
    }
    __syncthreads();
  }
}

int launch_topk_peaks(const float* spectra, int num_rows, int M, int k, int* idx_out, float* val_out, cudaStream_t st) {
  if (!spectra || !idx_out || M < 1 || M > 128 * kTopkMaxPerThread || k < 1 || k > M || num_rows < 0) return EIMS_ERR_ARG;
  if (num_rows == 0) return 0;
  const int blocks = num_rows < 148 * 16 ? num_rows : 148 * 16;
  launch_pdl(topk_peaks_kernel, dim3(blocks), dim3(128), 0, st, spectra, num_rows, M, k, idx_out, val_out);
  return 0;
}

// prob = sigmoid(logits) (inference) ; dlogits = dprob * p * (1-p) (autograd entry)
__global__ void sigmoid_kernel(const int* __restrict__ dims, const float* __restrict__ logits, int M,
                               float* __restrict__ prob, int early) {
  const int64_t n4 = (int64_t)pdl_sync_dims(dims, early).B * M / 4;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 u = ldg4(logits + 4 * i), p;
    p.x = 1.f / (1.f + expf(-u.x)); p.y = 1.f / (1.f + expf(-u.y));
    p.z = 1.f / (1.f + expf(-u.z)); p.w = 1.f / (1.f + expf(-u.w));
    st4(prob + 4 * i, p);
  }
}
__global__ void dprob_to_dlogits_kernel(const int* __restrict__ dims, const float* __restrict__ prob,
                                        const float* __restrict__ dprob, int M, float* __restrict__ dlogits) {
  pdl_sync();
  const int64_t n4 = (int64_t)dims[DIM_B] * M / 4;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 p = ldg4(prob + 4 * i), d = ldg4(dprob + 4 * i);
    d.x *= p.x * (1.f - p.x); d.y *= p.y * (1.f - p.y); d.z *= p.z * (1.f - p.z); d.w *= p.w * (1.f - p.w);
    st4(dlogits + 4 * i, d);
  }
}
static inline int ew_blocks(int64_t n4) {
  int64_t b = (n4 + 255) / 256;
  if (b > 148 * 8) b = 148 * 8;
  return b < 1 ? 1 : (int)b;
}
int launch_sigmoid(const int* dims, const float* logits, int M, float* prob, int max_graphs, cudaStream_t st) {
  launch_pdl(sigmoid_kernel, dim3(ew_blocks((int64_t)max_graphs * M / 4)), dim3(256), 0, st, dims, logits, M, prob, dims_early_ref());
  return 0;
}
int launch_dprob_to_dlogits(const int* dims, const float* prob, const float* dprob, int M, float* dlogits,
                            int max_graphs, cudaStream_t st) {
  launch_pdl(dprob_to_dlogits_kernel, dim3(ew_blocks((int64_t)max_graphs * M / 4)), dim3(256), 0, st, dims, prob, dprob, M, dlogits);
  return 0;
}

__global__ void __launch_bounds__(256) metrics_kernel(const int* __restrict__ dims, const float* __restrict__ row_loss,
                                                      const float* __restrict__ row_cos, int M,
                                                      float* __restrict__ metrics) {
  pdl_sync();
  metrics_reduce(dims[DIM_B], row_loss, row_cos, M, metrics);
}
int launch_metrics(const int* dims, const float* row_loss, const float* row_cos, int M, float* metrics, cudaStream_t st) {
  launch_pdl(metrics_kernel, dim3(1), dim3(256), 0, st, dims, row_loss, row_cos, M, metrics);
  return 0;
}

// =========================================================================== column sums (bias grads)
// out[c] += sum_r in[r,c]  for r < dims[dim_slot]
__global__ void __launch_bounds__(256) colsum_kernel(const int* __restrict__ dims, int dim_slot,
                                                     const float* __restrict__ in, int C, int ld, float* __restrict__ out, int early) {
  __shared__ float4 sh[4][64];
  const BatchDims bd = pdl_sync_dims(dims, early);
  const int R = dim_slot == DIM_B ? bd.B : (dim_slot == DIM_N ? bd.N : bd.E);
  const int cg = blockIdx.x * 64 + (threadIdx.x & 63), rs = threadIdx.x >> 6;
  const int rows_per = (R + gridDim.y - 1) / gridDim.y;
  const int r0 = blockIdx.y * rows_per, r1 = min(R, r0 + rows_per);
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  if (4 * cg < C)
    for (int r = r0 + rs; r < r1; r += 4) {
      float4 v = ldg4(in + (int64_t)r * ld + 4 * cg);
      a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
    }
  sh[rs][threadIdx.x & 63] = a;
  __syncthreads();
  if (rs == 0 && 4 * cg < C && r0 < r1) {
    for (int k = 1; k < 4; ++k) { float4 v = sh[k][threadIdx.x]; a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w; }
    atomicAdd(out + 4 * cg + 0, a.x); atomicAdd(out + 4 * cg + 1, a.y);
    atomicAdd(out + 4 * cg + 2, a.z); atomicAdd(out + 4 * cg + 3, a.w);
  }
}
int launch_colsum(const int* dims, int dim_slot, const float* in, int C, int ld, float* out, int max_rows, cudaStream_t st) {
  if (C % 4) return EIMS_ERR_ARG;
  int gy = (max_rows + 31) / 32;
  if (gy > 64) gy = 64;
  if (gy < 1) gy = 1;
  dim3 grid((C / 4 + 63) / 64, gy);
  launch_pdl(colsum_kernel, dim3(grid), dim3(256), 0, st, dims, dim_slot, in, C, ld, out, dims_early_ref());
  return 0;
}

// =========================================================================== K8 AdamW
// k_dev != null: the scalars come from the device-resident step block (captured CUDA graphs)
__global__ void __launch_bounds__(256) adamw_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m,
                                                    float* __restrict__ v, int64_t n, AdamK k, const AdamK* __restrict__ k_dev) {
  pdl_sync();
  if (k_dev) k = *k_dev;
  const int64_t n4 = n >> 2;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 pp = *reinterpret_cast<float4*>(p + 4 * i), gg = *reinterpret_cast<float4*>(g + 4 * i);
    float4 mm = *reinterpret_cast<float4*>(m + 4 * i), vv = *reinterpret_cast<float4*>(v + 4 * i);
#define EIMS_ADAM1(P, G, Mm, V)                                       \
  {                                                                   \
    float gr = G * k.grad_scale;                                      \
    P *= k.decay;                                                     \
    Mm = Mm + (gr - Mm) * k.one_minus_b1;                             \
    V = V * k.b2 + k.one_minus_b2 * gr * gr;                          \
    float den = sqrtf(V) * k.inv_bc2_sqrt + k.eps;                    \
    P = P - k.step_size * (Mm / den);                                 \
  }
    EIMS_ADAM1(pp.x, gg.x, mm.x, vv.x) EIMS_ADAM1(pp.y, gg.y, mm.y, vv.y)
    EIMS_ADAM1(pp.z, gg.z, mm.z, vv.z) EIMS_ADAM1(pp.w, gg.w, mm.w, vv.w)
    *reinterpret_cast<float4*>(p + 4 * i) = pp;
    *reinterpret_cast<float4*>(m + 4 * i) = mm;
    *reinterpret_cast<float4*>(v + 4 * i) = vv;
    *reinterpret_cast<float4*>(g + 4 * i) = make_float4(0.f, 0.f, 0.f, 0.f);  // optimizer.zero_grad (GCN:414)
  }
  if (blockIdx.x == 0)
    for (int64_t i = (n4 << 2) + threadIdx.x; i < n; i += blockDim.x) {
      float P = p[i], G = g[i], Mm = m[i], V = v[i];
      EIMS_ADAM1(P, G, Mm, V)
      p[i] = P; m[i] = Mm; v[i] = V; g[i] = 0.f;
    }
}

int launch_adamw(float* p, float* g, float* m, float* v, int64_t n, const eims_step* s, cudaStream_t st, const StepBlock* blk) {
  if (!blk && (!s || s->step < 1)) return EIMS_ERR_ARG;
  const AdamK k = blk ? AdamK{} : make_adam_k(s);
  launch_pdl(adamw_kernel, dim3(ew_blocks(n / 4)), dim3(256), 0, st, p, g, m, v, n, k, blk ? &blk->adam : nullptr);
  return 0;
}

// ---- step block upload: consecutive blocks (see StepBlock in common.cuh) by value, one launch for up to kStepPack
__global__ void step_blocks_store_kernel(StepBlockPack v, StepBlock* __restrict__ dst, int n) {
  pdl_sync();
  if ((int)threadIdx.x < n) dst[threadIdx.x] = v.b[threadIdx.x];
}
int launch_step_blocks_store(const StepBlockPack& v, StepBlock* dst, int n, cudaStream_t st) {
  if (n < 1 || n > kStepPack) return EIMS_ERR_ARG;
  launch_pdl(step_blocks_store_kernel, dim3(1), dim3(32), 0, st, v, dst, n);
  return 0;
}

// =========================================================================== dropout mask (tests)
__global__ void dropout_mask_kernel(DropCfg d, int64_t n4, float* __restrict__ out) {
  pdl_sync();
  d = resolve_drop(d);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 m = drop_mask4(d, (uint64_t)i * 4);
    m.x = m.x != 0.f; m.y = m.y != 0.f; m.z = m.z != 0.f; m.w = m.w != 0.f;
    st4(out + 4 * i, m);
  }
}
int launch_dropout_mask(DropCfg d, int rows, int W, float* out, cudaStream_t st) {
  if (W % 4) return EIMS_ERR_ARG;
  int64_t n4 = (int64_t)rows * W / 4;
  launch_pdl(dropout_mask_kernel, dim3(ew_blocks(n4)), dim3(256), 0, st, d, n4, out);
  return 0;
}

}  // namespace eims

EIMS_TIMELINE_READER(dense)
