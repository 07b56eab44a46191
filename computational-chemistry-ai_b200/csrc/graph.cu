// K1 batched-graph CSR builder, layer-0 fused aggregate+transform, K2 normalised-adjacency
// SpMM, K5 readout.  Integer work is bit-exact with the reference's dgl.batch / GraphConv
// degree normalisation (SURVEY A.1); aggregation sums neighbours in ascending edge-id order
// with separate multiply and add roundings, i.e. the order torch's index_add_ uses on the CPU.
#include "common.cuh"
#include "launchers.h"

namespace eims {

// ------------------------------------------------------------------------------------ K1
// One launch, one warp per molecule (4 per block).  Every block first reduces the atom / edge
// counts of the whole batch (B is a few hundred to a few thousand, the tables sit in L2): the
// totals give the capacity check, the counts of the molecules before the block's own give its
// node / edge offsets - so there is no separate scan launch.  Then each warp writes its
// molecule: features, COO edge list in reference order, CSR by destination (ascending edge id
// inside a row), per-atom graph id, degree normalisation, and (a0 != null) the 6-wide layer-0
// aggregate a0 = A (x * c) of GraphConv (GCN:359, i = 0), which only needs the molecule itself.
// dims[DIM_ZERO_DEG] holds the sequence number of the last batch that had an isolated atom and
// dims[5] the current sequence number (no reset race between blocks).
constexpr int kK1Warps = 4;  // upper bound (shared-memory arrays); launch_csr_build uses 2 warps per block
constexpr int kMaxF0 = 8;

// Large batches (inference, thousands of molecules): the per-block batch reduction of the fused
// kernel below would cost O(B) per block, so one 1024-thread block scans the counts first
// (exclusive scan of atoms / directed edges per molecule -> gptr, eptr, dims) and the build
// kernel reads its offsets from there.
__global__ void __launch_bounds__(1024) k1_scan_kernel(const int64_t* __restrict__ node_ptr,
                                                       const int64_t* __restrict__ bond_ptr,
                                                       const int32_t* __restrict__ ids, int B, int max_nodes,
                                                       int max_edges, int* __restrict__ gptr, int* __restrict__ eptr,
                                                       int* __restrict__ rowptr, int* __restrict__ dims, int seq,
                                                       const StepBlock* __restrict__ blk) {
  pdl_sync();
  if (blk) { ids = blk->ids; seq = blk->k1_seq; }  // captured graph: this step's ids / sequence number
  __shared__ int wn[32], we[32];
  __shared__ int carry_n, carry_e;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  if (tid == 0) { carry_n = 0; carry_e = 0; }
  __syncthreads();
  for (int base = 0; base < B; base += 1024) {
    int g = base + tid, n = 0, e = 0;
    if (g < B) {
      int64_t id = ids ? (int64_t)ids[g] : (int64_t)g;
      n = (int)(node_ptr[id + 1] - node_ptr[id]);
      e = 2 * (int)(bond_ptr[id + 1] - bond_ptr[id]);
    }
    int in = n, ie = e;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int tn = __shfl_up_sync(0xffffffffu, in, o), te = __shfl_up_sync(0xffffffffu, ie, o);
      if (lane >= o) { in += tn; ie += te; }
    }
    if (lane == 31) { wn[w] = in; we[w] = ie; }
    __syncthreads();
    if (w == 0) {
      int a = wn[lane], b = we[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int ta = __shfl_up_sync(0xffffffffu, a, o), tb = __shfl_up_sync(0xffffffffu, b, o);
        if (lane >= o) { a += ta; b += tb; }
      }
      wn[lane] = a; we[lane] = b;  // inclusive over warps
    }
    __syncthreads();
    int off_n = carry_n + (w ? wn[w - 1] : 0) + in - n;
    int off_e = carry_e + (w ? we[w - 1] : 0) + ie - e;
    if (g < B) { gptr[g] = off_n; eptr[g] = off_e; }
    __syncthreads();
    if (tid == 0) { carry_n += wn[31]; carry_e += we[31]; }
    __syncthreads();
  }
  if (tid == 0) {
    int N = carry_n, E = carry_e;
    bool over = N > max_nodes || E > max_edges || N < 0 || E < 0;
    gptr[B] = N; eptr[B] = E;
    dims[DIM_B] = over ? 0 : B;
    dims[DIM_N] = over ? 0 : N;
    dims[DIM_E] = over ? 0 : E;
    dims[DIM_OVERFLOW] = over ? 1 : 0;
    dims[5] = seq;
    dims[6] = dims[7] = 0;
    rowptr[over ? 0 : N] = over ? 0 : E;
  }
}

constexpr int kK1MaxN = 128, kK1MaxB = 192;  // molecule size staged in shared memory (bigger ones use global scratch)

struct K1Stage {  // per-warp staging
  int sb[kK1MaxB], se[kK1MaxB];   // bond ends (molecule-local)
  int scol[2 * kK1MaxB];          // CSR columns (molecule-local source atom)
  int srow[kK1MaxN + 1];          // row starts (molecule-local edge offset)
  int scnt[kK1MaxN];              // per-atom counters of the counting sort (degree, then fill cursor)
  float snorm[kK1MaxN];
  float sx[kK1MaxN * kMaxF0];
};

__global__ void __launch_bounds__(kK1Warps * 32) k1_build_kernel(
    const int64_t* __restrict__ node_ptr, const int64_t* __restrict__ bond_ptr, const float* __restrict__ feat,
    const int32_t* __restrict__ bond_begin, const int32_t* __restrict__ bond_end, const int32_t* __restrict__ ids, int B,
    int F, int max_nodes, int max_edges, int seq, int* __restrict__ gptr, int* __restrict__ eptr, int* __restrict__ gid,
    int* __restrict__ src, int* __restrict__ dst, int* __restrict__ rowptr, int* __restrict__ col,
    float* __restrict__ norm, float* __restrict__ x, float* __restrict__ a0, int* __restrict__ dims, int prescanned,
    const StepBlock* __restrict__ blk, int* __restrict__ bids) {
  pdl_sync();
  if (blk) { ids = blk->ids; seq = blk->k1_seq; }  // captured graph: this step's ids / sequence number
  __shared__ long long red[kK1Warps][4];
  __shared__ int cnt_n[kK1Warps], cnt_e[kK1Warps];
  __shared__ K1Stage stage[kK1Warps];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int nwarps = blockDim.x >> 5;   // warps (= molecules) per block
  const int g0 = blockIdx.x * nwarps;
  int o, eo;
  if (prescanned) {  // offsets and dims[] come from k1_scan_kernel
    if (dims[DIM_OVERFLOW]) return;
    const int g = g0 + w;
    if (g >= B) return;
    o = gptr[g]; eo = eptr[g];
    if (lane == 0) { cnt_n[w] = gptr[g + 1] - o; cnt_e[w] = eptr[g + 1] - eo; }
    __syncwarp();
  } else {
  // ---- phase A: batch totals and this block's prefix (loads batched 4 deep: the molecule
  // table is a random gather from HBM, so the two dependent latencies are paid once per batch)
  long long tn = 0, te = 0, pn = 0, pe = 0;
  for (int gb = threadIdx.x; gb < B; gb += 4 * blockDim.x) {
    int64_t id[4];
    long long n[4], e[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int g = gb + u * blockDim.x;
      id[u] = g < B ? (ids ? (int64_t)__ldg(ids + g) : (int64_t)g) : -1;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      n[u] = e[u] = 0;
      if (id[u] >= 0) {
        n[u] = __ldg(node_ptr + id[u] + 1) - __ldg(node_ptr + id[u]);
        e[u] = 2 * (__ldg(bond_ptr + id[u] + 1) - __ldg(bond_ptr + id[u]));
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int g = gb + u * blockDim.x;
      tn += n[u]; te += e[u];
      if (g < g0) { pn += n[u]; pe += e[u]; }
      if (g >= g0 && g < g0 + nwarps && g < B) { cnt_n[g - g0] = (int)n[u]; cnt_e[g - g0] = (int)e[u]; }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    tn += __shfl_xor_sync(0xffffffffu, tn, o); te += __shfl_xor_sync(0xffffffffu, te, o);
    pn += __shfl_xor_sync(0xffffffffu, pn, o); pe += __shfl_xor_sync(0xffffffffu, pe, o);
  }
  if (lane == 0) { red[w][0] = tn; red[w][1] = te; red[w][2] = pn; red[w][3] = pe; }
  __syncthreads();
  tn = te = pn = pe = 0;
  for (int k = 0; k < nwarps; ++k) { tn += red[k][0]; te += red[k][1]; pn += red[k][2]; pe += red[k][3]; }
  const bool over = tn > max_nodes || te > max_edges;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    const int N = over ? 0 : (int)tn, E = over ? 0 : (int)te;
    dims[DIM_B] = over ? 0 : B;
    dims[DIM_N] = N;
    dims[DIM_E] = E;
    dims[DIM_OVERFLOW] = over ? 1 : 0;
    dims[5] = seq;
    dims[6] = dims[7] = 0;
    if (!over) { gptr[B] = N; eptr[B] = E; }
    rowptr[N] = E;
  }
  if (over) return;
  if (g0 + w >= B) return;
  o = (int)pn; eo = (int)pe;
  for (int k = 0; k < w; ++k) { o += cnt_n[k]; eo += cnt_e[k]; }
  }
  const int g = g0 + w;
  // ---- phase B: this warp's molecule; every loop below is lane-parallel (atoms or edges
  // across lanes), the phases are separated by __syncwarp()
  const int64_t id = ids ? (int64_t)ids[g] : (int64_t)g;
  const int64_t a_0 = node_ptr[id], b_0 = bond_ptr[id];
  const int n = cnt_n[w], nb = cnt_e[w] >> 1, ne = 2 * nb;
  K1Stage& S = stage[w];
  const bool staged = n <= kK1MaxN && nb <= kK1MaxB;
  // molecule-local views: shared staging, or (oversized molecule) the global outputs themselves
  const int* pb = staged ? S.sb : bond_begin + b_0;
  const int* pe_ = staged ? S.se : bond_end + b_0;
  int* prow = staged ? S.srow : rowptr + o;
  int* pcol = staged ? S.scol : col + eo;
  float* pnorm = staged ? S.snorm : norm + o;
  const float* px = staged ? S.sx : x + (int64_t)o * F;
  const int rowbase = staged ? 0 : eo, colbase = staged ? 0 : o;
  if (lane == 0 && !prescanned) { gptr[g] = o; eptr[g] = eo; }
  if (lane == 0 && bids) bids[g] = (int)id;  // the batch's molecule ids = the target rows of the loss kernel
  for (int t = lane; t < n * F; t += 32) {
    const float v = __ldg(feat + a_0 * F + t);
    x[(int64_t)o * F + t] = v;
    if (staged) S.sx[t] = v;
  }
  for (int k = lane; k < nb; k += 32) {
    int bgn = __ldg(bond_begin + b_0 + k), end = __ldg(bond_end + b_0 + k);
    if ((unsigned)bgn >= (unsigned)n || (unsigned)end >= (unsigned)n) {  // corrupt table: flag it, stay in bounds
      dims[DIM_OVERFLOW] = 1;
      bgn = min(max(bgn, 0), n - 1);
      end = min(max(end, 0), n - 1);
    }
    if (staged) { S.sb[k] = bgn; S.se[k] = end; }
    src[eo + 2 * k] = o + bgn; dst[eo + 2 * k] = o + end;          // GCN:142-143: [b->e, e->b]
    src[eo + 2 * k + 1] = o + end; dst[eo + 2 * k + 1] = o + bgn;
  }
  __syncwarp();
  // ---- counting sort of the directed edges by destination, in shared memory (staged molecules):
  //   1. degree of every atom: one shared-memory atomic per bond end (lanes over bonds)
  //   2. row starts: exclusive warp scan of the degrees (lanes over atoms), degree normalisation
  //   3. every edge takes the next free slot of its destination row (lanes over edges, any order) ...
  //   4. ... and every row sorts its <= deg slots by edge id (lanes over atoms): ascending edge id inside a row,
  //      which is the order torch's index_add_ adds in.
  // Oversized molecules (beyond the staging arrays) keep the O(bonds) scans per atom / per edge on global memory.
  if (staged) {
    for (int i = lane; i < n; i += 32) S.scnt[i] = 0;
    __syncwarp();
    for (int k = lane; k < nb; k += 32) { atomicAdd(&S.scnt[S.sb[k]], 1); atomicAdd(&S.scnt[S.se[k]], 1); }
    __syncwarp();
  }
  int run = 0;
  for (int base = 0; base < n; base += 32) {
    const int i = base + lane;
    int deg = 0;
    if (i < n) {
      if (staged) { deg = S.scnt[i]; S.scnt[i] = 0; }  // the counter becomes the row's fill cursor
      else for (int k = 0; k < nb; ++k) deg += (pe_[k] == i) + (pb[k] == i);
    }
    int inc = deg;
#pragma unroll
    for (int sft = 1; sft < 32; sft <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, inc, sft);
      if (lane >= sft) inc += t;
    }
    const int total = __shfl_sync(0xffffffffu, inc, 31);
    if (i < n) {
      const int wpos = run + inc - deg;  // molecule-local
      // torch.pow(deg.float().clamp(min=1), -0.5) on the CPU == fl(1/fl(sqrt(d)))
      const float c = __fdiv_rn(1.0f, __fsqrt_rn((float)max(deg, 1)));
      rowptr[o + i] = eo + wpos;
      gid[o + i] = g;
      norm[o + i] = c;
      if (staged) { S.srow[i] = wpos; S.snorm[i] = c; }
      if (deg == 0) atomicMax(dims + DIM_ZERO_DEG, seq);
    }
    run += total;
  }
  if (staged && lane == 0) S.srow[n] = ne;
  __syncwarp();
  if (!staged) __threadfence_block();
  if (staged) {
    for (int e = lane; e < ne; e += 32) {   // edge e = 2k (b->e) or 2k+1 (e->b): destination = the other end
      const int k = e >> 1;
      const int d = (e & 1) ? S.sb[k] : S.se[k];
      S.scol[S.srow[d] + atomicAdd(&S.scnt[d], 1)] = e;
    }
    __syncwarp();
    for (int i = lane; i < n; i += 32) {
      const int a = S.srow[i], b = S.srow[i + 1];
      for (int x = a + 1; x < b; ++x) {     // insertion sort of the row's edge ids (deg is a handful)
        const int v = S.scol[x];
        int y = x - 1;
        while (y >= a && S.scol[y] > v) { S.scol[y + 1] = S.scol[y]; --y; }
        S.scol[y + 1] = v;
      }
      for (int x = a; x < b; ++x) {          // edge id -> source atom
        const int e = S.scol[x], k = e >> 1;
        const int sv = (e & 1) ? S.se[k] : S.sb[k];
        S.scol[x] = sv;
        col[eo + x] = o + sv;
      }
    }
  } else {
    // CSR columns (lane per directed edge): edge e lands in row dst(e) at the rank it has among the edges with the
    // same destination, i.e. in ascending edge id
    for (int e = lane; e < ne; e += 32) {
      const int k = e >> 1;
      const int d = (e & 1) ? pb[k] : pe_[k], sv = (e & 1) ? pe_[k] : pb[k];
      int rank = 0;
      for (int k2 = 0; k2 < k; ++k2) rank += (pe_[k2] == d) + (pb[k2] == d);
      if (e & 1) rank += (pe_[k] == d);  // edge 2k precedes edge 2k+1 (only matters for a self-bond)
      const int pos = prow[d] - rowbase + rank;  // molecule-local edge offset
      col[eo + pos] = o + sv;
    }
  }
  if (!a0) return;
  __syncwarp();
  if (!staged) __threadfence_block();
  // layer-0 aggregate (lane per atom): a0_i = sum_{j in row i} fl(x_j * c_j), ascending edge id,
  // separate multiply and add roundings (torch's CPU index_add_ order)
  for (int i = lane; i < n; i += 32) {
    float acc[kMaxF0];
#pragma unroll
    for (int f = 0; f < kMaxF0; ++f) acc[f] = 0.f;
    const int e0 = prow[i] - rowbase;
    const int e1 = (staged || i + 1 < n) ? prow[i + 1] - rowbase : ne;
    for (int e = e0; e < e1; ++e) {
      const int j = pcol[e] - colbase;
      const float cj = pnorm[j];
#pragma unroll
      for (int f = 0; f < kMaxF0; ++f)
        if (f < F) acc[f] = __fadd_rn(acc[f], __fmul_rn(px[j * F + f], cj));
    }
#pragma unroll
    for (int f = 0; f < kMaxF0; ++f)
      if (f < F) a0[(int64_t)(o + i) * F + f] = acc[f];
  }
}

int launch_csr_build(const eims_dataset* ds, const int32_t* ids, int B, int F, int max_nodes, int max_edges,
                     int* gptr, int* eptr, int* gid, int* src, int* dst, int* rowptr, int* col, float* norm,
                     float* x, int* dims, cudaStream_t st, float* a0, int seq, const StepBlock* blk, int* bids) {
  if (F > kMaxF0) return EIMS_ERR_ARG;
  // molecules (warps) per block: 2 gives 256 blocks for a batch of 512, 4 is round 1's shape
  constexpr int k1w = 2;
  static_assert(k1w <= kK1Warps, "k1_build_kernel is sized for at most kK1Warps warps");
  const int blocks = B > 0 ? (B + k1w - 1) / k1w : 1;
  const int prescanned = B > 1024;
  if (prescanned)
    launch_pdl(k1_scan_kernel, dim3(1), dim3(1024), 0, st, ds->node_ptr, ds->bond_ptr, ids, B, max_nodes, max_edges, gptr, eptr,
               rowptr, dims, seq, blk);
  launch_pdl(k1_build_kernel, dim3(blocks), dim3(k1w * 32), 0, st, ds->node_ptr, ds->bond_ptr, ds->feat, ds->bond_begin,
             ds->bond_end, ids, B, F, max_nodes, max_edges, seq, gptr, eptr, gid, src, dst, rowptr, col, norm, x, a0, dims,
             prescanned, blk, bids);
  return 0;
}

// --------------------------------------------------------------------------- layer 0 forward
// GraphConv(6 -> H) + ReLU (GCN:359-360 for i = 0) from the 6-wide aggregate a0 that K1 left:
// z0 = relu((a0 W0) * c + b0), the transform done in registers, with the BatchNorm statistics
// of z0 fused in (training).  Column-slab decomposition: grid = (H/64, row groups), thread =
// (4 columns, 1 of 16 row lanes).
constexpr int kL0Rows = 512;  // rows of a0 / norm a block stages in shared memory

__global__ void __launch_bounds__(256) layer0_fwd_kernel(const int* __restrict__ dims, const float* __restrict__ norm,
                                                         const float* __restrict__ a0, int F, const float* __restrict__ W,
                                                         const float* __restrict__ bias, int H, float* __restrict__ z,
                                                         BnFuse bn, float4* __restrict__ zero, int64_t zero_n4) {
  pdl_sync();
  // side job (training): zero the outputs of the split-K head GEMMs of this step
  if (zero) {
    const int64_t nth = (int64_t)gridDim.x * gridDim.y * blockDim.x;
    for (int64_t i = ((int64_t)blockIdx.y * gridDim.x + blockIdx.x) * blockDim.x + threadIdx.x; i < zero_n4; i += nth)
      zero[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  __shared__ float sa0[kL0Rows * kMaxF0];
  __shared__ float sc[kL0Rows];
  const int N = dims[DIM_N];
  const int cl = threadIdx.x & 15, rl = threadIdx.x >> 4;
  const int c0 = blockIdx.x * 64, c = c0 + cl * 4;
  // this block's contiguous row range (<= kL0Rows by construction of the grid)
  const int rpb = (N + gridDim.y - 1) / gridDim.y;
  const int r0 = blockIdx.y * rpb, r1 = min(N, r0 + rpb);
  const int nr = max(0, r1 - r0);
  for (int t = threadIdx.x; t < nr * F; t += blockDim.x) sa0[t] = __ldg(a0 + (int64_t)r0 * F + t);
  for (int t = threadIdx.x; t < nr; t += blockDim.x) sc[t] = __ldg(norm + r0 + t);
  __syncthreads();
  double sa[4] = {0.0, 0.0, 0.0, 0.0}, sb[4] = {0.0, 0.0, 0.0, 0.0};
  if (c < H) {
    float4 w[kMaxF0];
#pragma unroll
    for (int f = 0; f < kMaxF0; ++f) w[f] = f < F ? ldg4(W + (int64_t)f * H + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 b = ldg4(bias + c);
#pragma unroll 4
    for (int r = rl; r < nr; r += 16) {
      const float ci = sc[r];
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int f = 0; f < kMaxF0; ++f)
        if (f < F) {
          const float a = sa0[r * F + f];
          v.x = fmaf(a, w[f].x, v.x); v.y = fmaf(a, w[f].y, v.y); v.z = fmaf(a, w[f].z, v.z); v.w = fmaf(a, w[f].w, v.w);
        }
      v.x = fmaxf(fmaf(v.x, ci, b.x), 0.f); v.y = fmaxf(fmaf(v.y, ci, b.y), 0.f);
      v.z = fmaxf(fmaf(v.z, ci, b.z), 0.f); v.w = fmaxf(fmaf(v.w, ci, b.w), 0.f);
      st4(z + (int64_t)(r0 + r) * H + c, v);
      if (bn.acc) {
        const double x0 = v.x, x1 = v.y, x2 = v.z, x3 = v.w;
        sa[0] += x0; sa[1] += x1; sa[2] += x2; sa[3] += x3;
        sb[0] = fma(x0, x0, sb[0]); sb[1] = fma(x1, x1, sb[1]); sb[2] = fma(x2, x2, sb[2]); sb[3] = fma(x3, x3, sb[3]);
      }
    }
  }
  if (!bn.acc) return;
  __shared__ double red[16][2][64];
#pragma unroll
  for (int e = 0; e < 4; ++e) { red[rl][0][cl * 4 + e] = sa[e]; red[rl][1][cl * 4 + e] = sb[e]; }
  __syncthreads();
  if (threadIdx.x < 128) {
    const int which = threadIdx.x / 64, cc = threadIdx.x % 64;
    double t = 0.0;
#pragma unroll
    for (int r = 0; r < 16; ++r) t += red[r][which][cc];
    if (c0 + cc < H) atomicAdd(bn_acc_slot(bn.acc, H, blockIdx.y, which, c0 + cc), t);
  }
  if (last_block_ticket(bn.ticket, gridDim.x * gridDim.y)) bn_finalize(bn, N);
}

int launch_layer0_fwd(const int* dims, const float* norm, const float* a0, int F, const float* W, const float* bias,
                      int H, float* z, int max_nodes, cudaStream_t st, const BnFuse* bn, float* zero, int64_t zero_n4) {
  if (F > kMaxF0 || H % 4) return EIMS_ERR_ARG;
  const int slabs = (H + 63) / 64;
  // one wave: the kernel needs 104 registers, so two blocks are resident per SM (measured at cfg 2: 13.7 us with
  // 2 blocks per SM, 16.7-17.5 us with 3 or 4, i.e. a second wave)
  constexpr int kBlocksPerSm = 2;
  int rg = (148 * kBlocksPerSm + slabs - 1) / slabs;
  const int need = (max_nodes + kL0Rows - 1) / kL0Rows;  // a block stages at most kL0Rows rows
  if (rg < need) rg = need;
  if (rg < 1) rg = 1;
  launch_pdl(layer0_fwd_kernel, dim3(slabs, rg), dim3(256), 0, st, dims, norm, a0, F, W, bias, H, z, bn ? *bn : BnFuse{},
             reinterpret_cast<float4*>(zero), zero_n4);
  return 0;
}

// --------------------------------------------------------------------------- layer 0 backward to the atom features
// a0 = A D x and z0 = relu(D a0 W0 + b0), so with q0 = D (dz0 * relu') (the BatchNorm-backward apply pass stores it):
//   da0 = q0 W0^T   [N, F]                      (layer0_dgrad_kernel: warp per row, W0 staged in shared memory)
//   dx  = D A^T da0 = D A da0                  (feat_grad_kernel: every bond gives both directed edges, so A^T = A
//                                               and K1's CSR by destination is also the CSR by source)
__global__ void __launch_bounds__(256) layer0_dgrad_kernel(const int* __restrict__ dims, const float* __restrict__ q, int H,
                                                           const float* __restrict__ W0, int F, float* __restrict__ da0,
                                                           int early) {
  extern __shared__ __align__(16) float sw[];  // W0 [F][H]
  const int N = pdl_sync_dims(dims, early).N;
  for (int t = threadIdx.x; t < F * H; t += blockDim.x) sw[t] = __ldg(W0 + t);
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int i = warp; i < N; i += nwarps) {
    float acc[kMaxF0];
#pragma unroll
    for (int f = 0; f < kMaxF0; ++f) acc[f] = 0.f;
    for (int c = lane * 4; c < H; c += 128) {
      const float4 v = ldg4(q + (int64_t)i * H + c);
#pragma unroll
      for (int f = 0; f < kMaxF0; ++f)
        if (f < F) {
          const float4 w = *reinterpret_cast<const float4*>(sw + f * H + c);
          acc[f] = fmaf(v.x, w.x, fmaf(v.y, w.y, fmaf(v.z, w.z, fmaf(v.w, w.w, acc[f]))));
        }
    }
    float mine = 0.f;
#pragma unroll
    for (int f = 0; f < kMaxF0; ++f)
      if (f < F) {
        const float s = warp_sum(acc[f]);
        if (lane == f) mine = s;
      }
    if (lane < F) da0[(int64_t)i * F + lane] = mine;
  }
}

__global__ void __launch_bounds__(256) feat_grad_kernel(const int* __restrict__ dims, const int* __restrict__ rowptr,
                                                        const int* __restrict__ col, const float* __restrict__ norm,
                                                        const float* __restrict__ da0, int F, float* __restrict__ dx,
                                                        int early) {
  const int N = pdl_sync_dims(dims, early).N;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < N; j += gridDim.x * blockDim.x) {
    float acc[kMaxF0];
#pragma unroll
    for (int f = 0; f < kMaxF0; ++f) acc[f] = 0.f;
    const int e0 = __ldg(rowptr + j), e1 = __ldg(rowptr + j + 1);
    for (int e = e0; e < e1; ++e) {
      const int i = __ldg(col + e);
#pragma unroll
      for (int f = 0; f < kMaxF0; ++f)
        if (f < F) acc[f] += __ldg(da0 + (int64_t)i * F + f);
    }
    const float cj = __ldg(norm + j);
#pragma unroll
    for (int f = 0; f < kMaxF0; ++f)
      if (f < F) dx[(int64_t)j * F + f] = acc[f] * cj;
  }
}

int launch_layer0_dgrad(const int* dims, const float* q0, int H, const float* W0, int F, float* da0, int max_nodes,
                        cudaStream_t st) {
  if (F < 1 || F > kMaxF0 || H % 4 || H > 1024) return EIMS_ERR_ARG;
  int blocks = (max_nodes + 7) / 8;  // 8 warps, one row each
  if (blocks > 148 * 8) blocks = 148 * 8;
  launch_pdl(layer0_dgrad_kernel, dim3(blocks < 1 ? 1 : blocks), dim3(256), (size_t)F * H * sizeof(float), st, dims, q0, H,
             W0, F, da0, dims_early_ref());
  return 0;
}

int launch_feat_grad(const int* dims, const int* rowptr, const int* col, const float* norm, const float* da0, int F,
                     float* dx, int max_nodes, cudaStream_t st) {
  if (F < 1 || F > kMaxF0) return EIMS_ERR_ARG;
  int blocks = (max_nodes + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  launch_pdl(feat_grad_kernel, dim3(blocks < 1 ? 1 : blocks), dim3(256), 0, st, dims, rowptr, col, norm, da0, F, dx,
             dims_early_ref());
  return 0;
}

// ------------------------------------------------------------------------------------ K2
// Warp per destination row; lane owns NV float4 column groups (columns (i*32+lane)*4), so a
// whole row of H <= 128*NV floats is gathered by one warp-wide 128-bit load per neighbour and
// all NV*UE loads of a trip are independent (UE neighbours per trip).  Neighbours are added in
// ascending edge id, each with separate multiply and add roundings (torch's CPU index_add_).
//   forward  (out_mode 0): out_i = sum_j fl( drop(bn(h_j)) * c_j )
//   backward (out_mode 1): out_i = ( sum_j h_j ) * c_i * dropmask_i        (A symmetric)
// STATS (backward form only): the rows written are the dh of the BatchNorm below, so the kernel also
// produces that BatchNorm's backward statistics - column sums of dh and dh*xhat (fp32 over a warp's
// few rows, combined per block in shared memory, fp64 from there on) -> dgamma, dbeta and the two
// column means - which saves the separate statistics pass over dh and z.
template <int NV, int UE, bool STATS>
__global__ void __launch_bounds__(256) spmm_norm_kernel(const int* __restrict__ dims, const int* __restrict__ rowptr,
                                                        const int* __restrict__ col, const float* __restrict__ norm,
                                                        const float* __restrict__ h, int H,
                                                        const float* __restrict__ bn_scale,
                                                        const float* __restrict__ bn_shift, DropCfg drop, int out_mode,
                                                        float* __restrict__ out, int parts, BnBwdFuse bf, int early,
                                                        int64_t lo_off) {
  extern __shared__ float s_stats[];  // STATS: [warps per block][2][128 * NV]
  const int N = pdl_sync_dims(dims, early).N;
  // lo_off != 0: `out` is the hi plane of a stacked tf32 hi / lo pair (gemm_tma.cu), the lo plane lo_off floats
  // behind it; the rows up to the next multiple of 32 are zeroed (the weight gradient reduces over whole 32-row k-blocks)
  // (compiled out of the STATS instantiation, whose register count decides whether its one-wave grid fits: 80 vs 94)
  const int64_t lo = STATS ? (int64_t)0 : lo_off;
  const int Nw = lo ? ((N + 31) & ~31) : N;
  drop = resolve_drop(drop);
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const bool has_bn = bn_scale != nullptr;
  const bool in_drop = drop.active() && out_mode == 0;
  const bool out_drop = drop.active() && out_mode == 1;
  // `parts` warps share a row when H > 128*NV (warp = row*parts + part; part fixed per warp
  // because nwarps is a multiple of parts)
  const int cbase = (warp % parts) * (128 * NV);
  float4 sc[NV], sh[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const int c = cbase + (v * 32 + lane) * 4;
    sc[v] = make_float4(1.f, 1.f, 1.f, 1.f);
    sh[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (has_bn && c < H) { sc[v] = ldg4(bn_scale + c); sh[v] = ldg4(bn_shift + c); }
  }
  // (the BatchNorm's mean / invstd vectors are re-read per row - L1 hits - rather than held in 16 registers:
  // the gather needs the occupancy more)
  float4 s1[STATS ? NV : 1], s2[STATS ? NV : 1];
  if (STATS) {
#pragma unroll
    for (int v = 0; v < NV; ++v) s1[v] = s2[v] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  for (int i = warp / parts; i < Nw; i += nwarps / parts) {
    if (!STATS && i >= N) {
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        const int c = cbase + (v * 32 + lane) * 4;
        if (c >= H) continue;
        st4(out + (int64_t)i * H + c, make_float4(0.f, 0.f, 0.f, 0.f));
        st4(out + lo + (int64_t)i * H + c, make_float4(0.f, 0.f, 0.f, 0.f));
      }
      continue;
    }
    const int e0 = __ldg(rowptr + i), e1 = __ldg(rowptr + i + 1);
    float4 zrow[STATS ? NV : 1];
    if (STATS) {  // issued before the gather so that it is in flight with it
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        const int c = cbase + (v * 32 + lane) * 4;
        zrow[v] = c < H ? ldg4(bf.z + (int64_t)i * H + c) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    float4 acc[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int e = e0; e < e1; e += UE) {
      int j[UE];
      float cj[UE];
      float4 val[UE][NV];
#pragma unroll
      for (int u = 0; u < UE; ++u) j[u] = (e + u < e1) ? __ldg(col + e + u) : -1;
#pragma unroll
      for (int u = 0; u < UE; ++u) {
        cj[u] = (out_mode == 0 && j[u] >= 0) ? __ldg(norm + j[u]) : 1.f;
#pragma unroll
        for (int v = 0; v < NV; ++v) {
          const int c = cbase + (v * 32 + lane) * 4;
          val[u][v] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (j[u] >= 0 && c < H) val[u][v] = ldg4(h + (int64_t)j[u] * H + c);
        }
      }
#pragma unroll
      for (int u = 0; u < UE; ++u) {
        if (j[u] < 0) continue;
#pragma unroll
        for (int v = 0; v < NV; ++v) {
          const int c = cbase + (v * 32 + lane) * 4;
          if (c >= H) continue;
          float4 x = val[u][v];
          if (has_bn) {
            x.x = fmaf(x.x, sc[v].x, sh[v].x); x.y = fmaf(x.y, sc[v].y, sh[v].y);
            x.z = fmaf(x.z, sc[v].z, sh[v].z); x.w = fmaf(x.w, sc[v].w, sh[v].w);
          }
          if (in_drop) {
            const float4 m = drop_mask4(drop, (uint64_t)j[u] * H + c);
            x.x *= m.x; x.y *= m.y; x.z *= m.z; x.w *= m.w;
          }
          if (out_mode == 0) {
            x.x = __fmul_rn(x.x, cj[u]); x.y = __fmul_rn(x.y, cj[u]);
            x.z = __fmul_rn(x.z, cj[u]); x.w = __fmul_rn(x.w, cj[u]);
          }
          acc[v].x = __fadd_rn(acc[v].x, x.x); acc[v].y = __fadd_rn(acc[v].y, x.y);
          acc[v].z = __fadd_rn(acc[v].z, x.z); acc[v].w = __fadd_rn(acc[v].w, x.w);
        }
      }
    }
    const float ci = out_mode == 1 ? __ldg(norm + i) : 1.f;
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int c = cbase + (v * 32 + lane) * 4;
      if (c >= H) continue;
      float4 a = acc[v];
      if (out_mode == 1) {
        a.x *= ci; a.y *= ci; a.z *= ci; a.w *= ci;
        if (out_drop) {
          const float4 m = drop_mask4(drop, (uint64_t)i * H + c);
          a.x *= m.x; a.y *= m.y; a.z *= m.z; a.w *= m.w;
        }
      }
      if (!STATS && lo) {
        float4 hi4, lo4;
        split_tf32_planes4(a, hi4, lo4);
        st4(out + (int64_t)i * H + c, hi4);
        st4(out + lo + (int64_t)i * H + c, lo4);
      } else {
        st4(out + (int64_t)i * H + c, a);
      }
      if (STATS) {
        const float4 mu = ldg4(bf.mean + c), is = ldg4(bf.invstd + c);
        s1[v].x += a.x; s1[v].y += a.y; s1[v].z += a.z; s1[v].w += a.w;
        s2[v].x = fmaf(a.x, (zrow[v].x - mu.x) * is.x, s2[v].x); s2[v].y = fmaf(a.y, (zrow[v].y - mu.y) * is.y, s2[v].y);
        s2[v].z = fmaf(a.z, (zrow[v].z - mu.z) * is.z, s2[v].z); s2[v].w = fmaf(a.w, (zrow[v].w - mu.w) * is.w, s2[v].w);
      }
    }
  }
  if (STATS) {
    constexpr int CW = 128 * NV;  // columns per warp
    float* mine = s_stats + (threadIdx.x >> 5) * 2 * CW;
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      st4(mine + (v * 32 + lane) * 4, s1[v]);
      st4(mine + CW + (v * 32 + lane) * 4, s2[v]);
    }
    __syncthreads();
    const int wpb = blockDim.x >> 5;
    // fp32 atomics (these are plain sums - no cancellation as in a variance - and the L2 executes
    // fp32 reductions an order of magnitude faster than fp64 ones); the replicas are summed in fp64
    float* facc = reinterpret_cast<float*>(bf.acc);
    for (int k = threadIdx.x; k < 2 * H; k += blockDim.x) {
      const int which = k / H, cc = k % H, part = cc / CW, j = cc % CW;
      float t = 0.f;
      for (int w = part; w < wpb; w += parts) t += s_stats[(w * 2 + which) * CW + j];
      atomicAdd(facc + (size_t)(blockIdx.x % kBnReplicas) * 2 * H + k, t);
    }
    if (!last_block_ticket(bf.ticket, gridDim.x)) return;
    for (int k = threadIdx.x; k < H; k += blockDim.x) {
      double sa = 0.0, sb = 0.0;
#pragma unroll
      for (int r = 0; r < kBnReplicas; ++r) {
        float* q = facc + (size_t)r * 2 * H;
        sa += (double)__ldcg(q + k);
        sb += (double)__ldcg(q + H + k);
        q[k] = 0.f;
        q[H + k] = 0.f;
      }
      bf.dbeta[k] += (float)sa;
      bf.dgamma[k] += (float)sb;
      if (bf.means) {  // NULL in eval mode (see bn_bwd_stats_kernel)
        bf.means[k] = N > 0 ? (float)(sa / N) : 0.f;
        bf.means[H + k] = N > 0 ? (float)(sb / N) : 0.f;
      }
    }
  }
}

// ------------------------------------------------------------------------------------ K2, molecule tiles
// The same aggregation with the neighbour rows STAGED IN SHARED MEMORY.  A batched graph is block diagonal and K1
// lays the atoms of a molecule out contiguously, so everything row i of molecule g can reach is the contiguous
// [n_g, H] tile h[gptr[g] .. gptr[g+1]): one block takes one molecule at a time, brings the tile in with the bulk
// async-copy engine (cp.async.bulk global -> shared, completion on an mbarrier: ONE copy per molecule when the block
// owns all H columns, else one per row of its column chunk), applies the per-row transform (BatchNorm apply, dropout,
// source-side degree norm) ONCE per element in place, and sums the neighbours of every row out of shared memory.
// Against the gather kernel above: every row of h is read from L2 once instead of deg ~ 2.06 times, and the
// transform - the dropout hash made the forward gather instruction-issue bound - runs once per element instead of
// once per gathered element.  Same neighbour order, same roundings: bit-identical output.
// Molecules too large for the tile (n_g > cap_rows or more directed edges than cap_edges) take the gather path
// inside the same kernel.  STATS as above (backward form only).

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init1(uint32_t bar) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait_parity(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  const long long t0 = clock64();
  while (true) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    if (ok) break;
    if (clock64() - t0 > 4000000000LL) __trap();  // ~2 s: a protocol bug must not hang the GPU
  }
}

template <int NV, bool STATS, int THREADS>
__global__ void __launch_bounds__(THREADS) spmm_mol_kernel(const int* __restrict__ dims, const int* __restrict__ gptr,
                                                               const int* __restrict__ rowptr, const int* __restrict__ col,
                                                               const float* __restrict__ norm, const float* __restrict__ h, int H,
                                                               const float* __restrict__ bn_scale, const float* __restrict__ bn_shift,
                                                               DropCfg drop, int out_mode, float* __restrict__ out, int cap_rows,
                                                               int cap_edges, BnBwdFuse bf, int early, int64_t lo_off) {
  constexpr int HC = 128 * NV;  // columns a block owns
  extern __shared__ __align__(128) uint8_t mol_smem[];
  float* tile = reinterpret_cast<float*>(mol_smem);                    // [cap_rows][HC]
  int* scol = reinterpret_cast<int*>(tile + (size_t)cap_rows * HC);    // [cap_edges] molecule-local source rows
  int* srow = scol + cap_edges;                                        // [cap_rows + 1] molecule-local edge offsets
  float* snorm = reinterpret_cast<float*>(srow + cap_rows + 1);        // [cap_rows]
  float* s_stats = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(snorm + cap_rows) + 15) & ~(uintptr_t)15);  // STATS: [8 warps][2][HC]
  __shared__ __align__(8) uint64_t bar_storage;
  const uint32_t bar = smem_addr(&bar_storage);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) mbar_init1(bar);
  __syncthreads();
  const BatchDims bd = pdl_sync_dims(dims, early);
  drop = resolve_drop(drop);
  const int B = bd.B, N = bd.N;
  const int c0 = blockIdx.y * HC;
  const bool has_bn = bn_scale != nullptr;
  const bool in_drop = drop.active() && out_mode == 0;
  const bool out_drop = drop.active() && out_mode == 1;
  float4 sc[NV], sh[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const int c = c0 + (v * 32 + lane) * 4;
    sc[v] = make_float4(1.f, 1.f, 1.f, 1.f);
    sh[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (has_bn && c < H) { sc[v] = ldg4(bn_scale + c); sh[v] = ldg4(bn_shift + c); }
  }
  // the transform pass maps threads to columns differently: float4 column tq of the chunk, fixed per thread
  const int tq = tid % (HC / 4);
  float4 ta = make_float4(1.f, 1.f, 1.f, 1.f), tb = make_float4(0.f, 0.f, 0.f, 0.f);
  if (has_bn && c0 + tq * 4 < H) { ta = ldg4(bn_scale + c0 + tq * 4); tb = ldg4(bn_shift + c0 + tq * 4); }
  float4 s1[STATS ? NV : 1], s2[STATS ? NV : 1];
  if (STATS) {
#pragma unroll
    for (int v = 0; v < NV; ++v) s1[v] = s2[v] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  uint32_t phase = 0;
  for (int g = blockIdx.x; g < B; g += gridDim.x) {
    const int r0 = __ldg(gptr + g), r1 = __ldg(gptr + g + 1), n = r1 - r0;
    if (n <= 0) continue;
    const int e0 = __ldg(rowptr + r0), e1 = __ldg(rowptr + r1), ne = e1 - e0;
    const bool staged = n <= cap_rows && ne <= cap_edges;
    if (staged) {
      // ---- stage: the tile through the bulk-copy engine, the molecule's CSR slice through ordinary loads
      if (warp == 0) {
        if (H == HC) {  // the block owns whole rows: the tile is one contiguous range of h
          if (lane == 0) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // earlier generic accesses to the tile precede the async write
            mbar_expect_tx(bar, (uint32_t)n * HC * 4u);
            bulk_g2s(smem_addr(tile), h + (size_t)r0 * H, (uint32_t)n * HC * 4u, bar);
          }
        } else {
          if (lane == 0) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            mbar_expect_tx(bar, (uint32_t)n * HC * 4u);
          }
          __syncwarp();
          for (int i = lane; i < n; i += 32) bulk_g2s(smem_addr(tile + (size_t)i * HC), h + (size_t)(r0 + i) * H + c0, HC * 4u, bar);
        }
      }
      for (int e = tid; e < ne; e += THREADS) scol[e] = __ldg(col + e0 + e) - r0;
      for (int i = tid; i <= n; i += THREADS) srow[i] = __ldg(rowptr + r0 + i) - e0;
      for (int i = tid; i < n; i += THREADS) snorm[i] = __ldg(norm + r0 + i);
      mbar_wait_parity(bar, phase);
      phase ^= 1u;
      if (out_mode == 0) {
        __syncthreads();  // snorm visible
        // ---- transform in place, once per element: fl( drop(bn(h_j)) * c_j ).  A thread keeps one float4 column
        // (THREADS is a multiple of HC/4) and walks down the rows.
        for (int j = tid / (HC / 4); j < n; j += THREADS / (HC / 4)) {
          float4 x = *reinterpret_cast<float4*>(tile + (size_t)j * HC + tq * 4);
          if (has_bn) {
            x.x = fmaf(x.x, ta.x, tb.x); x.y = fmaf(x.y, ta.y, tb.y); x.z = fmaf(x.z, ta.z, tb.z); x.w = fmaf(x.w, ta.w, tb.w);
          }
          if (in_drop) {
            const float4 m = drop_mask4(drop, (uint64_t)(r0 + j) * H + c0 + tq * 4);
            x.x *= m.x; x.y *= m.y; x.z *= m.z; x.w *= m.w;
          }
          const float cj = snorm[j];
          x.x = __fmul_rn(x.x, cj); x.y = __fmul_rn(x.y, cj); x.z = __fmul_rn(x.z, cj); x.w = __fmul_rn(x.w, cj);
          *reinterpret_cast<float4*>(tile + (size_t)j * HC + tq * 4) = x;
        }
      }
      __syncthreads();
    }
    // ---- aggregate: warp per destination row, neighbours in ascending edge id
    for (int i = warp; i < n; i += THREADS / 32) {
      const int row = r0 + i;
      float4 zrow[STATS ? NV : 1];
      if (STATS) {
#pragma unroll
        for (int v = 0; v < NV; ++v) {
          const int c = c0 + (v * 32 + lane) * 4;
          zrow[v] = c < H ? ldg4(bf.z + (int64_t)row * H + c) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
      float4 acc[NV];
#pragma unroll
      for (int v = 0; v < NV; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (staged) {
        const int a0 = srow[i], a1 = srow[i + 1];
        for (int e = a0; e < a1; ++e) {
          const float* src = tile + (size_t)scol[e] * HC;
#pragma unroll
          for (int v = 0; v < NV; ++v) {
            const float4 x = *reinterpret_cast<const float4*>(src + (v * 32 + lane) * 4);
            acc[v].x = __fadd_rn(acc[v].x, x.x); acc[v].y = __fadd_rn(acc[v].y, x.y);
            acc[v].z = __fadd_rn(acc[v].z, x.z); acc[v].w = __fadd_rn(acc[v].w, x.w);
          }
        }
      } else {  // oversized molecule: gather from global, transform on the fly (as spmm_norm_kernel does)
        const int a0 = __ldg(rowptr + row), a1 = __ldg(rowptr + row + 1);
        for (int e = a0; e < a1; ++e) {
          const int j = __ldg(col + e);
          const float cj = out_mode == 0 ? __ldg(norm + j) : 1.f;
#pragma unroll
          for (int v = 0; v < NV; ++v) {
            const int c = c0 + (v * 32 + lane) * 4;
            if (c >= H) continue;
            float4 x = ldg4(h + (int64_t)j * H + c);
            if (has_bn) {
              x.x = fmaf(x.x, sc[v].x, sh[v].x); x.y = fmaf(x.y, sc[v].y, sh[v].y);
              x.z = fmaf(x.z, sc[v].z, sh[v].z); x.w = fmaf(x.w, sc[v].w, sh[v].w);
            }
            if (in_drop) {
              const float4 m = drop_mask4(drop, (uint64_t)j * H + c);
              x.x *= m.x; x.y *= m.y; x.z *= m.z; x.w *= m.w;
            }
            if (out_mode == 0) {
              x.x = __fmul_rn(x.x, cj); x.y = __fmul_rn(x.y, cj); x.z = __fmul_rn(x.z, cj); x.w = __fmul_rn(x.w, cj);
            }
            acc[v].x = __fadd_rn(acc[v].x, x.x); acc[v].y = __fadd_rn(acc[v].y, x.y);
            acc[v].z = __fadd_rn(acc[v].z, x.z); acc[v].w = __fadd_rn(acc[v].w, x.w);
          }
        }
      }
      const float ci = out_mode == 1 ? (staged ? snorm[i] : __ldg(norm + row)) : 1.f;
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        const int c = c0 + (v * 32 + lane) * 4;
        if (c >= H) continue;
        float4 a = acc[v];
        if (out_mode == 1) {
          a.x *= ci; a.y *= ci; a.z *= ci; a.w *= ci;
          if (out_drop) {
            const float4 m = drop_mask4(drop, (uint64_t)row * H + c);
            a.x *= m.x; a.y *= m.y; a.z *= m.z; a.w *= m.w;
          }
        }
        if (!STATS && lo_off) {  // stacked tf32 hi / lo planes (see spmm_norm_kernel)
          float4 hi4, lo4;
          split_tf32_planes4(a, hi4, lo4);
          st4(out + (int64_t)row * H + c, hi4);
          st4(out + lo_off + (int64_t)row * H + c, lo4);
        } else {
          st4(out + (int64_t)row * H + c, a);
        }
        if (STATS) {
          const float4 mu = ldg4(bf.mean + c), is = ldg4(bf.invstd + c);
          s1[v].x += a.x; s1[v].y += a.y; s1[v].z += a.z; s1[v].w += a.w;
          s2[v].x = fmaf(a.x, (zrow[v].x - mu.x) * is.x, s2[v].x); s2[v].y = fmaf(a.y, (zrow[v].y - mu.y) * is.y, s2[v].y);
          s2[v].z = fmaf(a.z, (zrow[v].z - mu.z) * is.z, s2[v].z); s2[v].w = fmaf(a.w, (zrow[v].w - mu.w) * is.w, s2[v].w);
        }
      }
    }
    __syncthreads();  // everyone is done with the tile and the index arrays before the next molecule overwrites them
  }
  if (!STATS && lo_off && blockIdx.x == 0) {  // rows [N, next multiple of 32) of both planes: zero (k-blocks of the weight gradient)
    const int Nw = (N + 31) & ~31;
    for (int k = tid; k < (Nw - N) * (HC / 4); k += THREADS) {
      const int row = N + k / (HC / 4), c = c0 + (k % (HC / 4)) * 4;
      if (c >= H) continue;
      st4(out + (int64_t)row * H + c, make_float4(0.f, 0.f, 0.f, 0.f));
      st4(out + lo_off + (int64_t)row * H + c, make_float4(0.f, 0.f, 0.f, 0.f));
    }
  }
  if (STATS) {
    // combine the block's warps in shared memory, one fp32 atomic per column and statistic into one of the
    // replicas, finalise in the last block of the whole grid (same scheme as spmm_norm_kernel<.., true>)
    float* mine = s_stats + warp * 2 * HC;
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      st4(mine + (v * 32 + lane) * 4, s1[v]);
      st4(mine + HC + (v * 32 + lane) * 4, s2[v]);
    }
    __syncthreads();
    float* facc = reinterpret_cast<float*>(bf.acc);
    for (int k = tid; k < 2 * HC; k += THREADS) {   // this block's column chunk
      const int which = k / HC, cc = k % HC;
      if (c0 + cc >= H) continue;
      float t = 0.f;
      for (int w = 0; w < THREADS / 32; ++w) t += s_stats[(w * 2 + which) * HC + cc];
      atomicAdd(facc + (size_t)(blockIdx.x % kBnReplicas) * 2 * H + (size_t)which * H + c0 + cc, t);
    }
    if (!last_block_ticket(bf.ticket, gridDim.x * gridDim.y)) return;
    for (int k = tid; k < H; k += THREADS) {
      double sa = 0.0, sb = 0.0;
#pragma unroll
      for (int r = 0; r < kBnReplicas; ++r) {
        float* q = facc + (size_t)r * 2 * H;
        sa += (double)__ldcg(q + k);
        sb += (double)__ldcg(q + H + k);
        q[k] = 0.f;
        q[H + k] = 0.f;
      }
      bf.dbeta[k] += (float)sa;
      bf.dgamma[k] += (float)sb;
      if (bf.means) {  // NULL in eval mode (see bn_bwd_stats_kernel)
        bf.means[k] = N > 0 ? (float)(sa / N) : 0.f;
        bf.means[H + k] = N > 0 ? (float)(sb / N) : 0.f;
      }
    }
  }
}

int launch_spmm_mol(const int* dims, const int* gptr, const int* rowptr, const int* col, const float* norm, const float* h,
                           int H, const float* bn_scale, const float* bn_shift, DropCfg drop, int out_mode, float* out,
                           int max_graphs, int tile_rows, cudaStream_t st, const BnBwdFuse* bf, int64_t lo_off) {
  // Shape: a block owns HC = 256 columns (8 warps) of one molecule at a time where H is a multiple of 256 and the
  // tile_rows x 1 KB tile fits in 64 KB (up to 64 rows), else HC = 128 columns (4 warps).
  const int NV = (H % 256 == 0 && (size_t)tile_rows * 256 * 4 <= 64 * 1024) ? 2 : 1;
  const int HC = 128 * NV, threads = 128 * NV;
  if (H % HC) return EIMS_ERR_ARG;
  const int cap_edges = 4 * tile_rows + 64;
  size_t smem = (size_t)tile_rows * HC * 4 + (size_t)cap_edges * 4 + (size_t)(tile_rows + 1) * 4 + (size_t)tile_rows * 4;
  smem = (smem + 15) & ~(size_t)15;
  if (bf) smem += (size_t)(threads / 32) * 2 * HC * 4;
  int gx = max_graphs < 1 ? 1 : max_graphs;
  const int chunks = H / HC;
  const int cap = 148 * 16 / chunks;   // grid-stride beyond a few waves (inference batches)
  if (gx > cap) gx = cap > 0 ? cap : 1;
  const BnBwdFuse none{};
#define EIMS_MOL(NVv, ST)                                                                                                   \
  do {                                                                                                                      \
    static bool attr = false;                                                                                               \
    if (!attr) { cudaFuncSetAttribute(spmm_mol_kernel<NVv, ST, 128 * NVv>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); attr = true; } \
    launch_pdl(spmm_mol_kernel<NVv, ST, 128 * NVv>, dim3(gx, chunks), dim3(128 * NVv), smem, st, dims, gptr, rowptr, col, norm, h, H, bn_scale, \
               bn_shift, drop, out_mode, out, tile_rows, cap_edges, bf ? *bf : none, dims_early_ref(), lo_off);             \
  } while (0)
  if (NV == 2) { if (bf) EIMS_MOL(2, true); else EIMS_MOL(2, false); }
  else { if (bf) EIMS_MOL(1, true); else EIMS_MOL(1, false); }
#undef EIMS_MOL
  return 0;
}

int launch_spmm_norm(const int* dims, const int* rowptr, const int* col, const float* norm, const float* h, int H,
                     const float* bn_scale, const float* bn_shift, DropCfg drop, int out_mode, float* out,
                     int max_nodes, cudaStream_t st, const BnBwdFuse* bf, const int* gptr, int max_graphs, int tile_rows,
                     int64_t lo_off) {
  if (H % 4) return EIMS_ERR_ARG;
  if (bf && (out_mode != 1 || H > 256)) return EIMS_ERR_ARG;  // the statistics form exists up to 256 columns (see plan.cu)
  if (lo_off && (bf || (lo_off & 3))) return EIMS_ERR_ARG;
  // Molecule-tile kernel (neighbour rows staged in shared memory by the bulk-copy engine) when the caller knows the
  // batch's graph offsets AND the batch is large.  Measured on a B200 (profiles/r2_spmm_ab.md): with >= ~8 molecules
  // per resident block (inference batches of 4096) staging wins, 0.128 vs 0.144 ms for the two cfg-3 launches (67 %
  // vs 59 % of the measured copy bandwidth); at a training batch of 512 molecules a block sees one molecule, its
  // phases (offsets -> bulk copy lands -> transform -> sum) cannot overlap, and the gather kernel - 9.5 k warps with
  // independent rows in flight - is faster (17 vs 18-26 us per launch for three staged variants, software-pipelined
  // producer/consumer ring included).
  const bool big_batch = max_graphs >= 2048 && !bf;
  if (big_batch && gptr && tile_rows > 0 && H % 128 == 0)
    return launch_spmm_mol(dims, gptr, rowptr, col, norm, h, H, bn_scale, bn_shift, drop, out_mode, out, max_graphs, tile_rows, st, bf, lo_off);
  const int parts = H <= 512 ? 1 : (H + 511) / 512;
  if (parts > 8 || (8 % parts)) return EIMS_ERR_ARG;  // 8 warps per block must split evenly over a row
  constexpr int kBlocksPerSm = 8;  // resident blocks per SM the grid is sized for
  int blocks = (max_nodes * parts + 7) / 8;
  if (blocks > 148 * kBlocksPerSm) blocks = 148 * kBlocksPerSm;
  if (blocks < 1) blocks = 1;
  // STATS: one wave of three blocks per SM (77 registers with one neighbour in flight per trip; measured at cfg 2:
  // 20 us with 444 blocks, 25 with 296 or 592)
  constexpr int kStatsBlocks = 148 * 3;
  const int blocks_s = blocks < kStatsBlocks ? blocks : kStatsBlocks;
#define EIMS_SPMM_STATS(NV)                                                                                            \
  launch_pdl(spmm_norm_kernel<NV, 1, true>, dim3(blocks_s), dim3(256), (size_t)8 * 2 * 128 * NV * sizeof(float), st, dims, rowptr, \
             col, norm, h, H, bn_scale, bn_shift, drop, out_mode, out, parts, *bf, dims_early_ref(), (int64_t)0)
#define EIMS_SPMM(NV, UE)                                                                                              \
  launch_pdl(spmm_norm_kernel<NV, UE, false>, dim3(blocks), dim3(256), 0, st, dims, rowptr, col, norm, h, H, bn_scale,  \
             bn_shift, drop, out_mode, out, parts, BnBwdFuse{}, dims_early_ref(), lo_off)
  if (bf) {
    if (H <= 128) EIMS_SPMM_STATS(1);
    else EIMS_SPMM_STATS(2);
  } else {
    if (H <= 128) EIMS_SPMM(1, 4);
    else if (H <= 256) EIMS_SPMM(2, 2);
    else EIMS_SPMM(4, 1);
  }
#undef EIMS_SPMM_STATS
#undef EIMS_SPMM
  return 0;
}

// ------------------------------------------------------------------------------------ K5
// Block per graph: BN apply + segment sum / mean / max / sum||max with the first arg-max
// (DGL's CPU SegmentCmp keeps the first maximum in node order).  256 threads = H/4 float4
// column lanes x (1024/H) row lanes; row lane k takes nodes r0+k, r0+k+RL, ... and the row
// lanes are combined in shared memory (ties between lanes go to the smaller node id).
__global__ void __launch_bounds__(256) readout_kernel(const int* __restrict__ dims, const int* __restrict__ gptr,
                                                      const float* __restrict__ z, int H,
                                                      const float* __restrict__ bn_scale,
                                                      const float* __restrict__ bn_shift, int pooling,
                                                      float* __restrict__ out, int* __restrict__ argmax,
                                                      float* __restrict__ zstat, const float* __restrict__ bn_mean,
                                                      int tile_bytes, int early) {
  extern __shared__ __align__(128) uint8_t ro_smem[];  // the graph's [n_g, H] tile of z when it fits tile_bytes
  __shared__ __align__(8) uint64_t bar_storage;
  __shared__ float4 ssum[256], smax[256], szs[256];
  __shared__ int4 sarg[256];
  const uint32_t bar = smem_addr(&bar_storage);
  if (threadIdx.x == 0 && tile_bytes > 0) mbar_init1(bar);
  __syncthreads();
  const int B = pdl_sync_dims(dims, early).B;
  const int g = blockIdx.x;
  if (g >= B) return;
  const int cpl = H >> 2;                       // float4 columns per row
  const int CL = cpl < 256 ? cpl : 256;         // column lanes
  const int RL = 256 / CL;                      // row lanes
  const int cl = threadIdx.x % CL, rl = threadIdx.x / CL;
  const int pool_dim = pooling == EIMS_POOL_COMBINED ? 2 * H : H;
  const bool has_bn = bn_scale != nullptr;
  const int r0 = __ldg(gptr + g), r1 = __ldg(gptr + g + 1);
  const float ninf = -__int_as_float(0x7f800000);
  // The graph's rows are contiguous: one bulk async copy brings the whole tile into shared memory and the row
  // lanes then stride over it there instead of issuing a chain of dependent L2 loads each (n_g / RL deep).
  const bool staged = tile_bytes > 0 && r1 > r0 && (int64_t)(r1 - r0) * H * 4 <= (int64_t)tile_bytes;
  const float* zt = z;          // row i of the graph is at zt + i * H
  const uint32_t tile_sa = smem_addr(ro_smem);
  if (staged) {
    if (threadIdx.x == 0) {
      mbar_expect_tx(bar, (uint32_t)(r1 - r0) * H * 4u);
      bulk_g2s(smem_addr(ro_smem), z + (int64_t)r0 * H, (uint32_t)(r1 - r0) * H * 4u, bar);
    }
    mbar_wait_parity(bar, 0);
    zt = reinterpret_cast<const float*>(ro_smem) - (int64_t)r0 * H;
  }
  for (int cb = 0; cb < cpl; cb += CL) {
    const int c = (cb + cl) * 4;
    const bool on = rl < RL && cb + cl < cpl;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f), mx = make_float4(ninf, ninf, ninf, ninf);
    float4 zs = make_float4(0.f, 0.f, 0.f, 0.f);  // column sums of (z - batch mean) over the graph, for zstat
    float4 mu = make_float4(0.f, 0.f, 0.f, 0.f);
    int4 am = make_int4(r0, r0, r0, r0);
    if (on) {
      float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
      if (has_bn) { sc = ldg4(bn_scale + c); sh = ldg4(bn_shift + c); }
      if (zstat) mu = ldg4(bn_mean + c);
#pragma unroll 4
      for (int i = r0 + rl; i < r1; i += RL) {
        float4 v;
        if (staged) {  // explicit shared-space load (through the generic pointer zt this is LD.E, several times the latency of LDS)
          const uint32_t sa = tile_sa + (uint32_t)((i - r0) * H + c) * 4u;
          asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(sa) : "memory");
        } else {
          v = ldg4(z + (int64_t)i * H + c);
        }
        zs.x += v.x - mu.x; zs.y += v.y - mu.y; zs.z += v.z - mu.z; zs.w += v.w - mu.w;
        v.x = fmaf(v.x, sc.x, sh.x); v.y = fmaf(v.y, sc.y, sh.y);
        v.z = fmaf(v.z, sc.z, sh.z); v.w = fmaf(v.w, sc.w, sh.w);
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
        if (v.x > mx.x) { mx.x = v.x; am.x = i; }
        if (v.y > mx.y) { mx.y = v.y; am.y = i; }
        if (v.z > mx.z) { mx.z = v.z; am.z = i; }
        if (v.w > mx.w) { mx.w = v.w; am.w = i; }
      }
    }
    __syncthreads();
    ssum[threadIdx.x] = s; smax[threadIdx.x] = mx; sarg[threadIdx.x] = am; szs[threadIdx.x] = zs;
    __syncthreads();
    if (rl == 0 && on) {
      for (int k = 1; k < RL; ++k) {
        const float4 s2 = ssum[k * CL + cl], m2 = smax[k * CL + cl];
        const int4 a2 = sarg[k * CL + cl];
        const float4 z2 = szs[k * CL + cl];
        zs.x += z2.x; zs.y += z2.y; zs.z += z2.z; zs.w += z2.w;
        s.x += s2.x; s.y += s2.y; s.z += s2.z; s.w += s2.w;
        if (m2.x > mx.x || (m2.x == mx.x && a2.x < am.x)) { mx.x = m2.x; am.x = a2.x; }
        if (m2.y > mx.y || (m2.y == mx.y && a2.y < am.y)) { mx.y = m2.y; am.y = a2.y; }
        if (m2.z > mx.z || (m2.z == mx.z && a2.z < am.z)) { mx.z = m2.z; am.z = a2.z; }
        if (m2.w > mx.w || (m2.w == mx.w && a2.w < am.w)) { mx.w = m2.w; am.w = a2.w; }
      }
      float* o = out + (int64_t)g * pool_dim;
      if (pooling == EIMS_POOL_MEAN) {
        const float n = (float)(r1 - r0);  // torch: S / n
        s.x = s.x / n; s.y = s.y / n; s.z = s.z / n; s.w = s.w / n;
      }
      if (pooling == EIMS_POOL_SUM || pooling == EIMS_POOL_MEAN || pooling == EIMS_POOL_COMBINED) st4(o + c, s);
      if (pooling == EIMS_POOL_MAX) st4(o + c, mx);
      if (pooling == EIMS_POOL_COMBINED) st4(o + H + c, mx);
      if (argmax && (pooling == EIMS_POOL_MAX || pooling == EIMS_POOL_COMBINED))
        *reinterpret_cast<int4*>(argmax + (int64_t)g * H + c) = am;
      if (zstat) {
        // what the BatchNorm-backward statistics of this layer need per graph (bn_bwd_stats_top_kernel):
        // the column sums of z - mean (summed centred, so nearly constant columns keep their digits) and
        // z - mean at the arg-max node
        float* zo = zstat + (int64_t)g * 2 * H;
        st4(zo + c, zs);
        if (r1 > r0)
          st4(zo + H + c, make_float4(zt[(int64_t)am.x * H + c] - mu.x, zt[(int64_t)am.y * H + c + 1] - mu.y,
                                      zt[(int64_t)am.z * H + c + 2] - mu.z, zt[(int64_t)am.w * H + c + 3] - mu.w));
      }
    }
  }
}

int launch_readout(const int* dims, const int* gptr, const float* z, int H, const float* bn_scale,
                   const float* bn_shift, int pooling, float* out, int* argmax, int max_graphs, cudaStream_t st, float* zstat,
                   const float* bn_mean) {
  if (H % 4 || H < 4 || (zstat && !bn_mean)) return EIMS_ERR_ARG;
  // shared-memory tile for the graph's rows (bulk async copy): 64 KB holds 64 atoms at H = 256; graphs that do not
  // fit read their rows from global memory
  constexpr int kTileBytes = 64 * 1024;
  const int tile_bytes = (H * 4) % 16 == 0 ? kTileBytes : 0;
  static bool attr = false;
  if (!attr) { cudaFuncSetAttribute(readout_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); attr = true; }
  launch_pdl(readout_kernel, dim3(max_graphs < 1 ? 1 : max_graphs), dim3(256), (size_t)tile_bytes, st, dims, gptr, z, H, bn_scale, bn_shift,
             pooling, out, argmax, zstat, bn_mean, tile_bytes, dims_early_ref());
  return 0;
}

}  // namespace eims

EIMS_TIMELINE_READER(graph)
