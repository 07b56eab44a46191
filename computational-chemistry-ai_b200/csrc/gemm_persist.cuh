// Pieces shared by the two persistent GEMM kernels (gemm_tma.cu: operands as pre-split planes by TMA; gemm_tc.cu: fp32
// operands split by producer warps): the device-side deal of work items to CTAs and the straight-line tile epilogue.
#pragma once
#include "common.cuh"

namespace eims {
namespace pg {

constexpr int BM = 128, BN = 256, BK = 32;
constexpr int kEpiWarps = 4;
constexpr int kPatchFloats = 32 * 36;   // padded 32 x 32 staging patch per epilogue warp
constexpr int kStatCols = 128;          // BatchNorm partial sums are flushed per half tile
constexpr int kMaxKbPerItem = 16;       // single accumulator per item: K <= 512 (see gemm_tc.cu)

__device__ __forceinline__ void mbar_arrive_local(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }

// explicit shared-space accesses for the epilogue's staging patch and statistics: through a pointer derived from the
// rounded-up dynamic shared-memory base the compiler emits GENERIC loads / stores (LD.E / ST.E instead of LDS / STS),
// measured ~45 cycles more per dependent access in a lone epilogue warp
__device__ __forceinline__ void sts_f4(uint32_t saddr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float4 lds_f4(uint32_t saddr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr) : "memory");
  return v;
}
__device__ __forceinline__ void sts_f64(uint32_t saddr, double v) {
  asm volatile("st.shared.f64 [%0], %1;" ::"r"(saddr), "d"(v) : "memory");
}
__device__ __forceinline__ double lds_f64(uint32_t saddr) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(saddr) : "memory");
  return v;
}

__device__ __forceinline__ void red_add_v4(float* p, float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// The share of CTA (pair) c of G (PAIR = 1: CTAs, PAIR = 2: CTA pairs) of the launch: identical in every role and in
// both CTAs of a pair, a pure function of the live sizes.  TM = rows of an output tile = 128 * PAIR.  Host-callable, so
// that the deal can be checked exhaustively without a GPU (tests/native/gemm_sched_probe.cu).
struct Sched {
  int ps, pk;                          // index of the store / the split-K problem, -1 = none
  int tiles_s, nt_s, kb_s;             // store problem: live tiles, column tiles, k-blocks per tile
  int KB, nt_k;                        // split-K problem: live k-blocks, column tiles
  int u0, u1;                          // this unit's k-block range of the split-K problem (tile-major index)
  int c, G;                            // index of this CTA (pair) and their number
};
struct Item { int prob, m0, n0, kb0, nkb; };
struct Cursor { int j, u; };

// what the schedule needs to know about the launch (each kernel fills it from its own parameter struct)
struct SchedIn { int nprob, ovh; int red[2], N[2]; };

template <int PAIR>
__host__ __device__ __forceinline__ Sched make_sched(const SchedIn& in, const int (&Mv)[2], const int (&Kv)[2], int c, int G) {
  constexpr int TM = BM * PAIR;
  Sched s;
  s.ps = s.pk = -1;
  for (int k = 0; k < in.nprob; ++k) {
    if (in.red[k]) s.pk = k; else s.ps = k;
  }
  s.c = c; s.G = G;
  s.tiles_s = 0; s.nt_s = 1; s.kb_s = 0; s.KB = 0; s.nt_k = 1; s.u0 = s.u1 = 0;
  if (s.ps >= 0) {
    s.nt_s = in.N[s.ps] / BN;
    s.tiles_s = ((Mv[s.ps] + TM - 1) / TM) * s.nt_s;
    s.kb_s = (Kv[s.ps] + BK - 1) / BK;
  }
  if (s.pk >= 0) {
    s.nt_k = in.N[s.pk] / BN;
    s.KB = (Kv[s.pk] + BK - 1) / BK;
    // (32-bit arithmetic: the host checks that units * CTAs stays far below 2^31; 64-bit divisions cost ~1 k cycles here)
    const int U = ((Mv[s.pk] + TM - 1) / TM) * s.nt_k * s.KB;
    const int t = s.tiles_s / G, r = s.tiles_s % G;
    const int cost = s.kb_s + in.ovh;
    // units [0, r) carry t + 1 store tiles, the others t: level the total (store cost + split-K k-blocks)
    const int T = (U + r * (t + 1) * cost + (G - r) * t * cost) / G;
    int x_hi = T - (t + 1) * cost;
    if (x_hi < 0) x_hi = 0;
    if (r * x_hi > U) x_hi = U / (r > 0 ? r : 1);
    const int rest = U - r * x_hi;
    if (c < r) {
      s.u0 = c * x_hi;
      s.u1 = s.u0 + x_hi;
    } else {
      const int nlo = G - r, j = c - r;
      s.u0 = r * x_hi + (int)((unsigned)rest * (unsigned)j / (unsigned)nlo);
      s.u1 = r * x_hi + (int)((unsigned)rest * (unsigned)(j + 1) / (unsigned)nlo);
    }
  }
  return s;
}

template <int PAIR>
__host__ __device__ __forceinline__ bool next_item(const Sched& s, Cursor& cur, Item& it) {
  constexpr int TM = BM * PAIR;
  if (s.ps >= 0) {
    const int t = s.c + cur.j * s.G;
    if (t < s.tiles_s && s.kb_s > 0) {
      ++cur.j;
      it.prob = s.ps; it.m0 = (t / s.nt_s) * TM; it.n0 = (t % s.nt_s) * BN; it.kb0 = 0; it.nkb = s.kb_s;
      return true;
    }
  }
  if (s.pk >= 0 && cur.u < s.u1) {
    const int tile = cur.u / s.KB, kb0 = cur.u % s.KB;
    int n = s.KB - kb0;
    if (n > s.u1 - cur.u) n = s.u1 - cur.u;
    if (n > kMaxKbPerItem) n = kMaxKbPerItem;
    it.prob = s.pk; it.m0 = (tile / s.nt_k) * TM; it.n0 = (tile % s.nt_k) * BN; it.kb0 = kb0; it.nkb = n;
    cur.u += n;
    return true;
  }
  return false;
}

// ---- epilogue of one 128 x 256 accumulator, per warp: its 32 rows in eight 32-column blocks.
// Straight-line code on purpose: an epilogue warp is alone on its scheduler, so every branch and every dependent
// latency is paid in full (the branchy version measured 1.4 k cycles per block, 14 k per tile).  Block cb + 1 is
// fetched from TMEM (tcgen05.ld, asynchronous) while block cb goes registers -> padded shared patch -> eight row
// segments of 128 bytes per store instruction.
struct EpiCtx {
  uint32_t patch, stats, taddr, release_bar;
  bool release_remote;
  int e, lane, et, m_q0, M, n0, ldc, bn_H;
  float rs, floor;
  float* Cq;            // C + (first row of this warp) * ldc + n0
  const float* bias;    // bias + n0 or null
  double* bn_acc;
};

__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// the registers are in / out operands so that nothing that uses them is scheduled above the wait
__device__ __forceinline__ void tmem_ld32_wait(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                 "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]),
                 "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]),
                 "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}

// VB = rows a thread has in flight between the patch read and the stores (8: all of its rows of the block, ~170
// registers; 4: two passes, fits the 96 registers a 21-warp CTA leaves per thread)
template <bool RED, bool STAT, bool FULL, bool DEEP, int VB = 8>
__device__ __forceinline__ void epilogue_tile(const EpiCtx& cx) {
  const int lane = cx.lane, cc = (lane & 7) * 4, r8 = lane >> 3;
  const uint32_t wr = cx.patch + lane * 144;                 // this thread's row of the patch (36 floats)
  const uint32_t rd = cx.patch + (r8 * 36 + cc) * 4;         // + t8 * 4 rows * 144 bytes
  float* const dst0 = cx.Cq + (int64_t)r8 * cx.ldc + cc;     // + t8 * 4 * ldc, + col0
  const int64_t step = (int64_t)4 * cx.ldc;
  uint32_t r[32];
  uint32_t rc[32];   // DEEP only (dead otherwise): the correction accumulator, 256 columns further
  tmem_ld32_issue(cx.taddr, r);
  if constexpr (DEEP) tmem_ld32_issue(cx.taddr + BN, rc);
  tmem_ld32_wait(r);
#pragma unroll 1
  for (int cb = 0; cb < BN / 32; ++cb) {
    const int col0 = cb * 32;
    if constexpr (DEEP) {
      tmem_ld32_wait(rc);
#pragma unroll
      for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(__uint_as_float(rc[j]) + __uint_as_float(r[j]));
    }
    __syncwarp();  // the previous block's reads of the patch are done
#pragma unroll
    for (int j = 0; j < 32; j += 4)
      sts_f4(wr + j * 4, make_float4(__uint_as_float(r[j]) * cx.rs, __uint_as_float(r[j + 1]) * cx.rs,
                                     __uint_as_float(r[j + 2]) * cx.rs, __uint_as_float(r[j + 3]) * cx.rs));
    __syncwarp();
    if (cb + 1 < BN / 32) {
      tmem_ld32_issue(cx.taddr + (uint32_t)(col0 + 32), r);   // in flight under the stores of this block
      if constexpr (DEEP) tmem_ld32_issue(cx.taddr + BN + (uint32_t)(col0 + 32), rc);
    } else {
      // the whole accumulator has left TMEM: hand the buffer back before the last block's stores
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) {
        if (cx.release_remote) mbar_arrive_cluster(cx.release_bar);
        else mbar_arrive_local(cx.release_bar);
      }
    }
    float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (cx.bias) b4 = ldg4(cx.bias + col0 + cc);
    float* dst = dst0 + col0;
    // column sums of the stored values (fp64, STAT only): this thread's 8 rows, then the four lanes that share a column quad
    double s1[4] = {0.0, 0.0, 0.0, 0.0}, s2[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int p = 0; p < 8; p += VB) {
      float4 v[VB];
#pragma unroll
      for (int t8 = 0; t8 < VB; ++t8) v[t8] = lds_f4(rd + (p + t8) * 4 * 144);
#pragma unroll
      for (int t8 = 0; t8 < VB; ++t8) {
        v[t8].x = fmaxf(v[t8].x + b4.x, cx.floor); v[t8].y = fmaxf(v[t8].y + b4.y, cx.floor);
        v[t8].z = fmaxf(v[t8].z + b4.z, cx.floor); v[t8].w = fmaxf(v[t8].w + b4.w, cx.floor);
      }
#pragma unroll
      for (int t8 = 0; t8 < VB; ++t8) {
        if (FULL || cx.m_q0 + (p + t8) * 4 + r8 < cx.M) {
          if (RED) red_add_v4(dst + (p + t8) * step, v[t8]);
          else st4(dst + (p + t8) * step, v[t8]);
          if (STAT) {
            const double d0 = v[t8].x, d1 = v[t8].y, d2 = v[t8].z, d3 = v[t8].w;
            s1[0] += d0; s1[1] += d1; s1[2] += d2; s1[3] += d3;
            s2[0] = fma(d0, d0, s2[0]); s2[1] = fma(d1, d1, s2[1]); s2[2] = fma(d2, d2, s2[2]); s2[3] = fma(d3, d3, s2[3]);
          }
        }
      }
    }
    if (STAT) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        s1[k] += __shfl_xor_sync(0xffffffffu, s1[k], 8);  s2[k] += __shfl_xor_sync(0xffffffffu, s2[k], 8);
        s1[k] += __shfl_xor_sync(0xffffffffu, s1[k], 16); s2[k] += __shfl_xor_sync(0xffffffffu, s2[k], 16);
      }
      const int sc = (cb & 3) * 32 + cc;  // column inside the half tile
      if (lane < 8) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          sts_f64(cx.stats + ((cx.e * 2 + 0) * kStatCols + sc + k) * 8, s1[k]);
          sts_f64(cx.stats + ((cx.e * 2 + 1) * kStatCols + sc + k) * 8, s2[k]);
        }
      }
      if ((cb & 3) == 3) {  // half a tile done: combine the four warps, one fp64 atomic per column and statistic
        asm volatile("bar.sync 1, 128;" ::: "memory");
#pragma unroll
        for (int which = 0; which < 2; ++which) {
          double t = 0.0;
#pragma unroll
          for (int w = 0; w < kEpiWarps; ++w) t += lds_f64(cx.stats + ((w * 2 + which) * kStatCols + cx.et) * 8);
          atomicAdd(bn_acc_slot(cx.bn_acc, cx.bn_H, blockIdx.x, which, cx.n0 + (cb >> 2) * kStatCols + cx.et), t);
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
      }
    }
    if (cb + 1 < BN / 32) tmem_ld32_wait(r);
  }
}

}  // namespace pg
}  // namespace eims
