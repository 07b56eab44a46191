// K3/K6: fp32-grade GEMM on the 5th-generation tensor cores (tcgen05.mma kind::tf32, fp32
// accumulators in TMEM), 3xTF32 split:  x = hi + lo with hi = rna_tf32(x), lo = rna_tf32(x - hi)
//   A*B ~= A_lo*B_hi + A_hi*B_lo + A_hi*B_hi       (the dropped lo*lo term is ~2^-22 relative)
// which is what the 1e-4 spectrum / gradient bar needs (single-pass TF32 gives 3e-3, SURVEY 7.3).
//
// Structure of one CTA (544 threads), one 128 x BN output tile:
//   warps 0-15 producers: 128-bit global loads of the fp32 A / B tiles (either storage order),
//              hi/lo split in registers, st.shared into the canonical UMMA SWIZZLE_128B layout
//              (K-major or MN-major, so no transposes anywhere), fence.proxy.async, one mbarrier
//              arrive per warp.  Two groups of 8 warps alternate k-blocks so two are in flight.
//              Interior tiles take a predicate-free path (thread-constant global / shared offsets,
//              one pointer bump per k-block); edge tiles and the K tail take the checked path.
//   warp  16   one elected lane issues 12 tcgen05.mma per k-block (4 k-steps x 3 products) and
//              tcgen05.commit's the stage back to the producers.
//   warps 0-15 epilogue: tcgen05.ld the accumulator (lane quarter = warp%4, 32-column slices by
//              warp/4) -> row scale -> shared staging tile -> bias / ReLU -> coalesced row stores
//              or red.global.add.v4.f32 (split-K).
// Sizes M and K may live in device memory (atoms in the current batch) so a captured step
// can be replayed; tiles past the live range exit before touching barriers or TMEM.

#include "common.cuh"
#include "gemm_persist.cuh"
#include "launchers.h"

namespace eims {

namespace tc {

// Optional pipeline trace (-DEIMS_GEMM_TRACE, tools/gemm_trace.py): SM-clock stamps of the phases
// of a few CTAs, to see where a tile's time goes.  Compiled out of the product library.
#ifdef EIMS_GEMM_TRACE
constexpr int kTraceCtas = 8, kTraceSlots = 128;
__device__ unsigned long long g_trace[kTraceCtas * kTraceSlots];
#define TRACE(slot)                                                                                   \
  do {                                                                                                \
    const int _c = blockIdx.x;                                                                        \
    if (_c < kTraceCtas && (threadIdx.x & 31) == 0) g_trace[_c * kTraceSlots + (slot)] = clock64();   \
  } while (0)
#else
#define TRACE(slot) do { } while (0)
#endif

constexpr int BM = 128, BK = 32;
constexpr int kProducerWarps = 16, kGroupThreads = 256, kThreads = (kProducerWarps + 1) * 32;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  const long long t0 = clock64();
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if (ok) break;
    if (clock64() - t0 > 4000000000LL) __trap();  // ~2 s: a protocol bug must not hang the GPU
  }
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
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
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// UMMA shared-memory matrix descriptor (sm_100 format, version 1).
// layout_type: 2 = SWIZZLE_128B (16-byte swizzle units), 1 = SWIZZLE_128B with 32-byte base
// (the only swizzled layout the hardware accepts for MN-major 32-bit / tf32 operands).
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
  d |= (uint64_t)layout_type << 61;
  return d;
}

// x = hi + lo with hi = rna_tf32(x), lo = rna_tf32(x - hi).  cvt.rna.tf32.f32 has no SASS
// instruction on sm_100 (it expands to a NaN/Inf test, an add, a select and a mask), so the
// round-to-nearest-away is done directly on the magnitude bits: +2^12, clear the 13 low bits.
// Identical to cvt.rna for every finite input (Inf stays Inf, NaN stays NaN).
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = (__float_as_uint(x) + 0x1000u) & 0xffffe000u;
  const float r = x - __uint_as_float(hi);
  lo = (__float_as_uint(r) + 0x1000u) & 0xffffe000u;
}

struct Args {
  const float* A; const float* B; float* C;
  int lda, ldb, ldc, a_mn, b_mn;
  int M, N, K;
  const int* m_dev; const int* k_dev;
  const float* row_scale; const float* bias;
  int relu, accumulate, vec_a, vec_b;
  int early;  // m_dev / k_dev (the batch's sizes) may be read before the grid-dependency wait (see pdl_sync_dims)
  int nt, mt, splits;  // tile grid of this problem: CTA `local` -> (local % nt, local / nt % mt, local / (nt * mt))
  BnFuse bn;  // bn.acc != null: column sums of the stored C (after bias / ReLU) -> BatchNorm statistics
};

// One launch runs up to two independent problems (a weight gradient and the data gradient that
// consume the same dy): CTAs [0, ctas0) work on g[0], the rest on g[1].
struct Group {
  Args g[2];
  int ctas0;
};

// Load one 16-byte chunk (4 consecutive floats) with zero fill outside [0, lim) of the
// contiguous dimension; `ok` gates the whole chunk (strided dimension in range).
__device__ __forceinline__ float4 load_chunk(const float* base, int64_t off, int pos, int lim, bool ok, int vec) {
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (!ok || pos >= lim) return v;
  const float* p = base + off;
  if (vec && pos + 3 < lim) return ldg4(p);
  v.x = __ldg(p);
  if (pos + 1 < lim) v.y = __ldg(p + 1);
  if (pos + 2 < lim) v.z = __ldg(p + 2);
  if (pos + 3 < lim) v.w = __ldg(p + 3);
  return v;
}

__device__ __forceinline__ void sts128(uint32_t saddr, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// explicit shared-space accesses for the epilogue's staging tile: through a pointer derived from the rounded-up dynamic
// shared-memory base the compiler emits GENERIC loads / stores (LD.E / ST.E instead of LDS / STS), ~4x the latency
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

__device__ __forceinline__ void store_split(uint32_t hi_saddr, uint32_t lo_saddr, float4 v) {
  uint4 h, l;
  split_tf32(v.x, h.x, l.x); split_tf32(v.y, h.y, l.y); split_tf32(v.z, h.z, l.z); split_tf32(v.w, h.w, l.w);
  sts128(hi_saddr, h);
  sts128(lo_saddr, l);
}

// Tile of an operand with ROWS "MN" rows and BK k-columns, written by one producer group
// (256 threads).  mn_major = 0: memory is [mn][k] (k contiguous) -> canonical K-major
// SWIZZLE_128B layout (8-row x 128-byte atoms, 16-byte chunk index XOR row%8):
//   offset(r, c) = (r/8)*1024 + (r%8)*128 + ((c ^ (r%8))*16)          c = 16-byte chunk along k
// mn_major = 1: memory is [k][mn] (mn contiguous) -> canonical MN-major SWIZZLE_128B_BASE32B
// layout (atoms of 4 k-rows x 128 bytes = 32 mn elements; 32-byte chunk index XOR k%4):
//   offset(k, c) = (k/4)*(ROWS/32*512) + (c/8)*512 + (k%4)*128 + ((((c%8)>>1) ^ (k%4))*32) + (c&1)*16
//   with c = 16-byte chunk along mn;  LBO = 512 (next 32 mn), SBO = ROWS/32*512 (next 4 k)
// Work split: chunk `it` of thread t.  K-major: chunk index it*256+t -> row = it*32 + t/8,
// c = t%8.  MN-major: one warp = one 512-byte atom (lanes 0-7 -> k-row 0, 8-15 -> k-row 1, ..),
// atom = it*8 + t/32.  In both layouts the shared offset is  soff(t) + it*4096  and the global
// element offset is  goff(t) + it*gstride,  which is what the predicate-free path uses.
// GT = threads that share one operand tile (a producer group of 8 warps)
template <int ROWS, int GT = kGroupThreads>
struct TileRegs {
  static constexpr int PER = ROWS * BK / 4 / GT;  // 16-byte chunks per producer thread
  float4 v[PER];
};

// (k, mn) element coordinates inside the tile of chunk `it` of thread t
template <int ROWS, int GT = kGroupThreads>
__device__ __forceinline__ void chunk_coords(int mn_major, int it, int t, int& mn, int& k) {
  if (!mn_major) {
    const int idx = it * GT + t;
    mn = idx >> 3;
    k = (idx & 7) * 4;
  } else {
    constexpr int MNA = ROWS / 32;  // mn atoms per 4-k-row group
    const int atom = it * (GT / 32) + (t >> 5);
    k = (atom / MNA) * 4 + ((t >> 3) & 3);
    mn = ((atom % MNA) * 8 + (t & 7)) * 4;
  }
}

// shared-memory byte offset of chunk 0 of thread t (chunk `it` is GT * 16 bytes further)
template <int ROWS>
__device__ __forceinline__ uint32_t chunk_soff(int mn_major, int t) {
  if (!mn_major) {
    const int row = t >> 3, c = t & 7;
    return (uint32_t)((row >> 3) * 1024 + (row & 7) * 128 + ((c ^ (row & 7)) << 4));
  }
  const int kk = (t >> 3) & 3, c = t & 7;
  return (uint32_t)((t >> 5) * 512 + kk * 128 + (((c >> 1) ^ kk) << 5) + ((c & 1) << 4));
}

// One operand as seen by one producer thread.
template <int ROWS, int GT = kGroupThreads>
struct Operand {
  const float* base;   // matrix origin
  const float* fast;   // pointer of chunk 0 of this thread in the group's current k-block
  int64_t kadv;        // elements between successive k-blocks of this thread's group (kb_stride k-blocks)
  int64_t gstride;     // elements between chunks it and it+1
  int ld, mn_major, vec, mn0, mn_lim, full;
  uint32_t soff;

  __device__ __forceinline__ void init(const float* b, int ld_, int mn_major_, int vec_, int mn0_, int mn_lim_, int kbeg,
                                       int t, int kb_stride = 2) {
    base = b; ld = ld_; mn_major = mn_major_; vec = vec_; mn0 = mn0_; mn_lim = mn_lim_;
    full = vec_ && (mn0_ + ROWS <= mn_lim_);
    int mn, k, mn1, k1;
    chunk_coords<ROWS, GT>(mn_major_, 0, t, mn, k);
    chunk_coords<ROWS, GT>(mn_major_, 1, t, mn1, k1);
    if (!mn_major_) {
      fast = b + (int64_t)(mn0_ + mn) * ld_ + kbeg + k;
      gstride = (int64_t)(mn1 - mn) * ld_;
      kadv = kb_stride * BK;
    } else {
      fast = b + (int64_t)(kbeg + k) * ld_ + mn0_ + mn;
      gstride = (int64_t)(k1 - k) * ld_ + (mn1 - mn);
      kadv = (int64_t)kb_stride * BK * ld_;
    }
    soff = chunk_soff<ROWS>(mn_major_, t);
  }

  // global -> registers for the k-block starting at k0 (issued early: the loads of a group's
  // next k-block are in flight while it waits for the stage to be released)
  __device__ __forceinline__ void load(TileRegs<ROWS, GT>& r, int k0, int k_lim, int t) {
    constexpr int PER = TileRegs<ROWS, GT>::PER;
    if (full && k0 + BK <= k_lim) {
      // MN-major with fewer atoms per pass than the tile is wide (8 producer warps on a 256-wide B tile): the passes
      // walk (mn atoms, then k-groups), two strides instead of one; all compile-time in `it`
      constexpr int API = GT / 32, MNA = ROWS / 32, R = API < MNA ? MNA / API : 1;
#pragma unroll
      for (int it = 0; it < PER; ++it) {
        const int64_t off = (mn_major && API < MNA) ? (int64_t)((it / R) * 4) * ld + (it % R) * API * 32 : it * gstride;
        r.v[it] = ldg4(fast + off);
      }
    } else {
#pragma unroll
      for (int it = 0; it < PER; ++it) {
        int mn, k;
        chunk_coords<ROWS, GT>(mn_major, it, t, mn, k);
        mn += mn0;
        k += k0;
        if (!mn_major) r.v[it] = load_chunk(base, (int64_t)mn * ld + k, k, k_lim, mn < mn_lim, vec);
        else r.v[it] = load_chunk(base, (int64_t)k * ld + mn, mn, mn_lim, k < k_lim, vec);
      }
    }
    fast += kadv;
  }

  // registers -> hi/lo split -> canonical UMMA shared-memory layout
  __device__ __forceinline__ void store(const TileRegs<ROWS, GT>& r, uint32_t hi_tile, uint32_t lo_tile) const {
    constexpr int PER = TileRegs<ROWS, GT>::PER;
#pragma unroll
    for (int it = 0; it < PER; ++it) store_split(hi_tile + soff + it * (GT * 16u), lo_tile + soff + it * (GT * 16u), r.v[it]);
  }
};

__device__ __forceinline__ void red_add_v4(float* p, float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

template <int BN, int STAGES>
__global__ void __launch_bounds__(kThreads, 1) gemm_3xtf32_kernel(const __grid_constant__ Group grp) {
  const int which = (int)blockIdx.x >= grp.ctas0 ? 1 : 0;
  const Args& g = grp.g[which];
  const int local = (int)blockIdx.x - (which ? grp.ctas0 : 0);
  const int bx = local % g.nt, by = (local / g.nt) % g.mt, bz = local / (g.nt * g.mt);
  constexpr int A_TILE = BM * BK * 4, B_TILE = BN * BK * 4;
  constexpr int STAGE_BYTES = 2 * A_TILE + 2 * B_TILE;
  // Two fp32 accumulators in TMEM: columns [0,BN) take the A_hi*B_hi products, columns [BN,2BN)
  // the two correction products.  The tensor core truncates (toward zero) every time it adds
  // into an accumulator - about half an ulp of the accumulator per MMA - so keeping the 2^-11
  // smaller corrections out of the main accumulator cuts that bias to a third (measured:
  // K = 1024, rms error 9e-6 -> 3e-6 of the mean |C|); the two are added in fp32 in the epilogue.
  // The 128-wide tile has TMEM to spare (512 columns per SM), so it also rotates the main
  // products over kMain = 3 accumulators: each then sees a third of the additions at a third of
  // the magnitude, which cuts the bias by another factor of three.
  constexpr int kMain = BN <= 128 ? 3 : 1;
  constexpr int kTmemCols = BN <= 128 ? 512 : 2 * BN;
  constexpr int kCorrCol = kMain * BN;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  __shared__ __align__(8) uint64_t bars[2 * STAGES + 1];
  __shared__ uint32_t tmem_base_slot;

  // Prologue that touches no global memory (barriers, TMEM) runs before the grid-dependency
  // wait, i.e. while the preceding kernel of the step is still draining.
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0) TRACE(0);
  const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[STAGES]), accum_bar = smem_u32(&bars[2 * STAGES]);
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(full0 + 8 * s, kGroupThreads / 32); mbar_init(empty0 + 8 * s, 1); }
    mbar_init(accum_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kProducerWarps) tmem_alloc(smem_u32(&tmem_base_slot), kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_slot;
  const uint32_t smem_base = smem_u32(smem);
  if (warp == 0) TRACE(1);
  int M = g.M, K = g.K;
  if (g.early) { if (g.m_dev) M = __ldcg(g.m_dev); if (g.k_dev) K = __ldcg(g.k_dev); }
  pdl_sync();
  if (warp == 0) TRACE(2);
  if (!g.early) { if (g.m_dev) M = __ldcg(g.m_dev); if (g.k_dev) K = __ldcg(g.k_dev); }
  const int N = g.N;
  const int m0 = by * BM, n0 = bx * BN;
  const int kblocks = (K + BK - 1) / BK;
  const int per_split = (kblocks + g.splits - 1) / g.splits;
  const int kb0 = bz * per_split;
  const int kb1 = min(kblocks, kb0 + per_split);
  const int nkb = kb1 - kb0;
  // dead tiles: past the live M (device-side size) or a split-K slice past the live K
  const bool live = m0 < M && n0 < N && nkb > 0;

  if (!live) {
    // nothing to do, but TMEM must still be released below
  } else
  if (warp < kProducerWarps) {
    // ---------------------------------------------------------------- producers
    const int group = warp >> 3, t = threadIdx.x & (kGroupThreads - 1);
    TileRegs<BM> ra;
    TileRegs<BN> rb;
    Operand<BM> oa;
    Operand<BN> ob;
    oa.init(g.A, g.lda, g.a_mn, g.vec_a, m0, M, (kb0 + group) * BK, t);
    ob.init(g.B, g.ldb, g.b_mn, g.vec_b, n0, N, (kb0 + group) * BK, t);
    if (group < nkb) {
      const int k0 = (kb0 + group) * BK;
      oa.load(ra, k0, K, t);
      ob.load(rb, k0, K, t);
    }
    for (int i = group; i < nkb; i += 2) {
      const int s = i % STAGES;
      const uint32_t ph = (uint32_t)(i / STAGES) & 1u;
      mbar_wait(empty0 + 8 * s, ph ^ 1u);
      if ((warp & 7) == 0 && i < 12) TRACE(8 + i * 4);
      const uint32_t st = smem_base + s * STAGE_BYTES;
      oa.store(ra, st, st + A_TILE);
      ob.store(rb, st + 2 * A_TILE, st + 2 * A_TILE + B_TILE);
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(full0 + 8 * s);
      if ((warp & 7) == 0 && i < 12) TRACE(8 + i * 4 + 1);
      if (i + 2 < nkb) {  // prefetch this group's next k-block while the tensor core works
        const int k0 = (kb0 + i + 2) * BK;
        oa.load(ra, k0, K, t);
        ob.load(rb, k0, K, t);
      }
    }
    // ---------------------------------------------------------------- epilogue
    // TMEM -> registers (row scale) -> shared staging tile (the pipeline stages are free once
    // the accumulator barrier has fired) -> bias / ReLU -> coalesced 512-byte row stores.
    mbar_wait(accum_bar, 0);
    tc_fence_after();
    if (warp == 0) TRACE(3);
    constexpr int LDS = BN + 4;  // padded row stride (floats): conflict-free float4 row writes
    const uint32_t stage = smem_base;  // shared-space byte address of the staging tile (the pipeline stages are free by now)
    {
      const int q = warp & 3;
      const int row = q * 32 + lane, m = m0 + row;
      const float rs = (g.row_scale && m < M) ? __ldg(g.row_scale + m) : 1.f;
#pragma unroll 1
      for (int col0 = (warp >> 2) * 32; col0 < BN; col0 += 128) {
        uint32_t r[32], c[32];
        const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)col0;
        tmem_ld32(lane_base + kCorrCol, r);  // smallest terms first
        const int used = min(kMain, nkb * (BK / 8));  // accumulators that received at least one MMA
#pragma unroll
        for (int a = kMain - 1; a >= 0; --a) {
          if (a < used) {
            tmem_ld32(lane_base + a * BN, c);
#pragma unroll
            for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) + __uint_as_float(c[j]));
          }
        }
        const uint32_t dst = stage + (uint32_t)(row * LDS + col0) * 4u;
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          sts_f4(dst + j * 4, make_float4(__uint_as_float(r[j]) * rs, __uint_as_float(r[j + 1]) * rs,
                                          __uint_as_float(r[j + 2]) * rs, __uint_as_float(r[j + 3]) * rs));
      }
    }
    tc_fence_before();
    asm volatile("bar.sync 1, 512;" ::: "memory");  // the 16 epilogue warps only
    if (warp == 0) TRACE(4);
    if (warp == 0) TRACE(5);
    {
      const bool add_bias = g.bias && (!g.accumulate || bz == 0);
      const bool vec_out = (g.ldc & 3) == 0 && ((reinterpret_cast<uintptr_t>(g.C) & 15) == 0);
      const bool stats = g.bn.acc != nullptr;
      // BatchNorm statistics of this tile ride on the store loop: a thread owns BN/128 column quads
      // and every 16th row, and keeps fp64 sums of what it stores (after bias / ReLU)
      constexpr int QUADS = BN / 128;
      double s1[QUADS][4], s2[QUADS][4];
#pragma unroll
      for (int qd = 0; qd < QUADS; ++qd)
#pragma unroll
        for (int e = 0; e < 4; ++e) s1[qd][e] = s2[qd][e] = 0.0;
#pragma unroll
      for (int qd = 0; qd < QUADS; ++qd) {
        const int c = 4 * lane + qd * 128;
        const int n = n0 + c;
        if (n >= N) break;
        float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (add_bias) {
          b4.x = __ldg(g.bias + n);
          if (n + 1 < N) b4.y = __ldg(g.bias + n + 1);
          if (n + 2 < N) b4.z = __ldg(g.bias + n + 2);
          if (n + 3 < N) b4.w = __ldg(g.bias + n + 3);
        }
        const bool v4 = vec_out && n + 3 < N;
#pragma unroll 4
        for (int row = warp; row < BM; row += kProducerWarps) {
          const int m = m0 + row;
          if (m >= M) break;
          float4 v = lds_f4(stage + (uint32_t)(row * LDS + c) * 4u);
          v.x += b4.x; v.y += b4.y; v.z += b4.z; v.w += b4.w;
          if (g.relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
          if (stats) {
            const double d0 = v.x, d1 = v.y, d2 = v.z, d3 = v.w;
            s1[qd][0] += d0; s1[qd][1] += d1; s1[qd][2] += d2; s1[qd][3] += d3;
            s2[qd][0] = fma(d0, d0, s2[qd][0]); s2[qd][1] = fma(d1, d1, s2[qd][1]);
            s2[qd][2] = fma(d2, d2, s2[qd][2]); s2[qd][3] = fma(d3, d3, s2[qd][3]);
          }
          float* dst = g.C + (int64_t)m * g.ldc + n;
          if (g.accumulate) {
            if (v4) {
              red_add_v4(dst, v);
            } else {
              atomicAdd(dst, v.x);
              if (n + 1 < N) atomicAdd(dst + 1, v.y);
              if (n + 2 < N) atomicAdd(dst + 2, v.z);
              if (n + 3 < N) atomicAdd(dst + 3, v.w);
            }
          } else if (v4) {
            st4(dst, v);
          } else {
            dst[0] = v.x;
            if (n + 1 < N) dst[1] = v.y;
            if (n + 2 < N) dst[2] = v.z;
            if (n + 3 < N) dst[3] = v.w;
          }
        }
      }
      if (stats) {
        // combine the 16 warps in shared memory (the staging tile is dead once every warp has read
        // its rows), then one fp64 atomic per column and statistic
        asm volatile("bar.sync 1, 512;" ::: "memory");
        const uint32_t red = smem_base;  // double [16 warps][2][BN]
#pragma unroll
        for (int qd = 0; qd < QUADS; ++qd)
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int c = 4 * lane + qd * 128 + e;
            sts_f64(red + (uint32_t)((warp * 2 + 0) * BN + c) * 8u, s1[qd][e]);
            sts_f64(red + (uint32_t)((warp * 2 + 1) * BN + c) * 8u, s2[qd][e]);
          }
        asm volatile("bar.sync 1, 512;" ::: "memory");
        for (int k = threadIdx.x; k < 2 * BN; k += kProducerWarps * 32) {
          const int which = k / BN, cc = k % BN;
          double tsum = 0.0;
#pragma unroll
          for (int w = 0; w < kProducerWarps; ++w) tsum += lds_f64(red + (uint32_t)((w * 2 + which) * BN + cc) * 8u);
          if (n0 + cc < N) atomicAdd(bn_acc_slot(g.bn.acc, g.bn.H, blockIdx.x, which, n0 + cc), tsum);
        }
      }
    }
  } else {
    // ---------------------------------------------------------------- MMA issuer
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)g.a_mn << 15) | ((uint32_t)g.b_mn << 16) |
                           ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
    // K-major: 8-row groups 1024 B apart (SBO); k-step (8 tf32) = +32 B inside the 128-B swizzle row.
    // MN-major: 32-element MN atoms 512 B apart (LBO); 4-row k-groups ROWS/32*512 B apart (SBO);
    //           k-step (8 k-rows = 2 k-groups) = +ROWS/32*1024 B.
    const uint32_t a_lbo = g.a_mn ? 512u : 16u, a_sbo = g.a_mn ? (uint32_t)(BM / 32 * 512) : 1024u;
    const uint32_t b_lbo = g.b_mn ? 512u : 16u, b_sbo = g.b_mn ? (uint32_t)(BN / 32 * 512) : 1024u;
    const uint32_t a_kstep = g.a_mn ? (uint32_t)(BM / 32 * 1024) : 32u;
    const uint32_t b_kstep = g.b_mn ? (uint32_t)(BN / 32 * 1024) : 32u;
    const uint32_t a_lt = g.a_mn ? 1u : 2u, b_lt = g.b_mn ? 1u : 2u;
    for (int i = 0; i < nkb; ++i) {
      const int s = i % STAGES;
      const uint32_t ph = (uint32_t)(i / STAGES) & 1u;
      mbar_wait(full0 + 8 * s, ph);
      tc_fence_after();
      if (i < 12) TRACE(8 + i * 4 + 2);
      if (lane == 0) {
        const uint32_t sa = smem_base + s * STAGE_BYTES;
        const uint32_t a_hi = sa, a_lo = sa + A_TILE, b_hi = sa + 2 * A_TILE, b_lo = b_hi + B_TILE;
#pragma unroll
        for (int ks = 0; ks < BK / 8; ++ks) {
          const uint64_t dah = make_desc(a_hi + ks * a_kstep, a_lbo, a_sbo, a_lt);
          const uint64_t dal = make_desc(a_lo + ks * a_kstep, a_lbo, a_sbo, a_lt);
          const uint64_t dbh = make_desc(b_hi + ks * b_kstep, b_lbo, b_sbo, b_lt);
          const uint64_t dbl = make_desc(b_lo + ks * b_kstep, b_lbo, b_sbo, b_lt);
          const int step = i * (BK / 8) + ks;  // k-step index inside this CTA's K range
          umma_tf32(tmem_base + kCorrCol, dal, dbh, idesc, step > 0 ? 1u : 0u);
          umma_tf32(tmem_base + kCorrCol, dah, dbl, idesc, 1u);
          umma_tf32(tmem_base + (step % kMain) * BN, dah, dbh, idesc, step >= kMain ? 1u : 0u);
        }
        umma_commit(empty0 + 8 * s);                 // frees the stage when these MMAs retire
        if (i == nkb - 1) umma_commit(accum_bar);    // accumulator complete
      }
      __syncwarp();
    }
    tc_fence_before();
  }
  if (warp == 0) TRACE(6);
  __syncthreads();
  if (warp == kProducerWarps) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
  if (g.bn.acc && live) {  // splits == 1 here; tiles past the live M are not counted
    const unsigned int live = (unsigned int)((M + BM - 1) / BM) * (unsigned int)g.nt;
    if (last_block_ticket(g.bn.ticket, live)) bn_finalize(g.bn, M);
  }
  if (warp == 0) TRACE(7);
}


// ---------------------------------------------------------------------------------------------
// Persistent variant: one CTA per SM walks over the 128 x 256 output tiles of one store problem with two 256-column
// accumulators in TMEM, so the epilogue of tile i runs under the main loop of tile i + 1.  Used for launches with several
// tiles per SM (inference forwards when the planes kernel of gemm_tma.cu is off); the tiles are dealt out on the device
// from the live row count (gemm_persist.cuh).
// A kernel that allocates tensor memory runs ONE CTA per SM on this driver (cudaOccupancyMaxActiveBlocksPerMultiprocessor
// says 1 for any kernel containing tcgen05.alloc, tools/ubench/occ_probe.cu), so overlap has to come from inside the CTA.
//   warps 0-7  : A tile of every k-block of the CTA's item sequence, warps 8-15: B tile (global -> registers, prefetched
//                one k-block ahead across item boundaries -> hi/lo split -> stage n & 1)
//   warps 16-19: epilogue (pg::epilogue_tile: straight-line, explicit shared-space patch, TMEM loads pipelined; the
//                first version of this kernel ran a branchy epilogue through generic pointers - LD.E / ST.E instead of
//                LDS / STS - which took 23 k cycles per tile instead of 5 k and hid the benefit of the overlap)
//   warp 20    : MMA issuer, all three products of a k-step into ONE accumulator (K <= 512 per item keeps the
//                accumulate-truncation bias at ~1e-6)
// (21 warps leave 96 registers per thread: the epilogue runs its rows in two passes of four (VB = 4).  With 8
// producer warps and the one-pass epilogue the main loop was producer-bound, 2.5 k instead of 1.9 k cycles per k-block;
// with 16 the epilogue warps starve for issue slots - see use_persistent().)
constexpr int kPersistProducerWarps = 16, kPersistGroupThreads = kPersistProducerWarps / 2 * 32;
constexpr int kPersistThreads = (kPersistProducerWarps + 1 + pg::kEpiWarps) * 32;
constexpr int kPersistStageBytes = 2 * BM * BK * 4 + 2 * 256 * BK * 4;
constexpr int kPersistOffPatch = 2 * kPersistStageBytes;
constexpr int kPersistOffStats = kPersistOffPatch + pg::kEpiWarps * pg::kPatchFloats * 4;
constexpr int kPersistSmem = kPersistOffStats + pg::kEpiWarps * 2 * pg::kStatCols * 8 + 1024;

// Producers: warps 0-7 bring the A tile (IS_B = false, ROWS = BM), warps 8-15 the B tile (ROWS = 256).  One operand per
// thread keeps the prefetched k-block at 16 / 32 registers.  `op_off` = byte offset of the operand's hi tile inside a
// stage; its lo tile follows it.
template <int ROWS, bool IS_B>
__device__ __forceinline__ void persistent_producer(const Args& g, const pg::Sched& sch, int M, int K, uint32_t smem_base,
                                                    uint32_t full0, uint32_t empty0, uint32_t op_off) {
  const int t = threadIdx.x & (kPersistGroupThreads - 1), lane = threadIdx.x & 31;
  TileRegs<ROWS, kPersistGroupThreads> regs;
  Operand<ROWS, kPersistGroupThreads> op;
  pg::Cursor cur{0, sch.u0};
  pg::Item it;
  int i = 0;
  auto enter = [&]() -> bool {
    if (!pg::next_item<1>(sch, cur, it)) return false;
    if (!IS_B) op.init(g.A, g.lda, g.a_mn, g.vec_a, it.m0, M, it.kb0 * BK, t, 1);
    else op.init(g.B, g.ldb, g.b_mn, g.vec_b, it.n0, g.N, it.kb0 * BK, t, 1);
    i = 0;
    return true;
  };
  bool valid = enter();
  if (valid) op.load(regs, it.kb0 * BK, K, t);
  uint32_t n = 0;
  while (valid) {
    const uint32_t sidx = n & 1u;
    mbar_wait(empty0 + 8 * sidx, ((n >> 1) & 1u) ^ 1u);
    const uint32_t hi = smem_base + sidx * kPersistStageBytes + op_off;
    op.store(regs, hi, hi + ROWS * BK * 4);
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) mbar_arrive(full0 + 8 * sidx);
    ++n;
    if (++i >= it.nkb) valid = enter();
    if (valid) op.load(regs, (it.kb0 + i) * BK, K, t);
  }
}

__global__ void __launch_bounds__(kPersistThreads, 1) gemm_3xtf32_persistent_kernel(const __grid_constant__ Args g) {
  constexpr int BN = 256;
  constexpr int A_TILE = BM * BK * 4, B_TILE = BN * BK * 4;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  __shared__ __align__(8) uint64_t bars[8];  // full[2], empty[2], acc_full[2], acc_empty[2]
  __shared__ uint32_t tmem_base_slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[2]), accf0 = smem_u32(&bars[4]), acce0 = smem_u32(&bars[6]);
  if (threadIdx.x == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(full0 + 8 * s, kPersistProducerWarps);
      mbar_init(empty0 + 8 * s, 1);
      mbar_init(accf0 + 8 * s, 1);
      mbar_init(acce0 + 8 * s, pg::kEpiWarps);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  constexpr int kMmaWarp = kPersistProducerWarps + pg::kEpiWarps;
  if (warp == kMmaWarp) tmem_alloc(smem_u32(&tmem_base_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_slot;
  const uint32_t smem_base = smem_u32(smem);
  int Mv[2] = {g.M, 0}, Kv[2] = {g.K, 0};
  if (g.early) { if (g.m_dev) Mv[0] = __ldcg(g.m_dev); if (g.k_dev) Kv[0] = __ldcg(g.k_dev); }
  pdl_sync();
  if (warp == 0) TRACE(0);
  if (!g.early) { if (g.m_dev) Mv[0] = __ldcg(g.m_dev); if (g.k_dev) Kv[0] = __ldcg(g.k_dev); }
  const int M = Mv[0], K = Kv[0];
  pg::SchedIn sin;
  sin.nprob = 1; sin.ovh = 0;   // one store problem: no split-K items to balance against
  sin.red[0] = sin.red[1] = 0; sin.N[0] = sin.N[1] = g.N;
  const pg::Sched sch = pg::make_sched<1>(sin, Mv, Kv);

  if (warp < kPersistProducerWarps) {
    // ---------------------------------------------------------------- producers
    if (warp < kPersistProducerWarps / 2) persistent_producer<BM, false>(g, sch, M, K, smem_base, full0, empty0, 0u);
    else persistent_producer<BN, true>(g, sch, M, K, smem_base, full0, empty0, 2u * A_TILE);
  } else if (warp == kMmaWarp) {
    // ---------------------------------------------------------------- MMA issuer
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)g.a_mn << 15) | ((uint32_t)g.b_mn << 16) |
                           ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
    const uint32_t a_lbo = g.a_mn ? 512u : 16u, a_sbo = g.a_mn ? (uint32_t)(BM / 32 * 512) : 1024u;
    const uint32_t b_lbo = g.b_mn ? 512u : 16u, b_sbo = g.b_mn ? (uint32_t)(BN / 32 * 512) : 1024u;
    const uint32_t a_kstep = g.a_mn ? (uint32_t)(BM / 32 * 1024) : 32u;
    const uint32_t b_kstep = g.b_mn ? (uint32_t)(BN / 32 * 1024) : 32u;
    const uint32_t a_lt = g.a_mn ? 1u : 2u, b_lt = g.b_mn ? 1u : 2u;
    pg::Cursor cur{0, sch.u0};
    pg::Item it;
    uint32_t n = 0, tcount = 0;
    while (pg::next_item<1>(sch, cur, it)) {
      const uint32_t b = tcount & 1u;
      if (tcount < 8) TRACE(16 + tcount * 8 + 0);
      mbar_wait(acce0 + 8 * b, ((tcount >> 1) & 1u) ^ 1u);  // accumulator b drained by the epilogue warps
      tc_fence_after();
      if (tcount < 8) TRACE(16 + tcount * 8 + 1);
      const uint32_t acc = tmem_base + b * BN;
      for (int i = 0; i < it.nkb; ++i, ++n) {
        const uint32_t s = n & 1u, ph = (n >> 1) & 1u;
        mbar_wait(full0 + 8 * s, ph);
        tc_fence_after();
        if (tcount < 8 && i == 0) TRACE(16 + tcount * 8 + 2);
        if (tcount < 8 && i == it.nkb - 1) TRACE(16 + tcount * 8 + 3);
        if (lane == 0) {
          const uint32_t sa = smem_base + s * kPersistStageBytes;
          const uint32_t a_hi = sa, a_lo = sa + A_TILE, b_hi = sa + 2 * A_TILE, b_lo = b_hi + B_TILE;
#pragma unroll
          for (int ks = 0; ks < BK / 8; ++ks) {
            const uint64_t dah = make_desc(a_hi + ks * a_kstep, a_lbo, a_sbo, a_lt);
            const uint64_t dal = make_desc(a_lo + ks * a_kstep, a_lbo, a_sbo, a_lt);
            const uint64_t dbh = make_desc(b_hi + ks * b_kstep, b_lbo, b_sbo, b_lt);
            const uint64_t dbl = make_desc(b_lo + ks * b_kstep, b_lbo, b_sbo, b_lt);
            umma_tf32(acc, dal, dbh, idesc, (i > 0 || ks > 0) ? 1u : 0u);
            umma_tf32(acc, dah, dbl, idesc, 1u);
            umma_tf32(acc, dah, dbh, idesc, 1u);
          }
          umma_commit(empty0 + 8 * s);                        // frees the stage when these MMAs retire
          if (i == it.nkb - 1) umma_commit(accf0 + 8 * b);    // accumulator b complete
        }
        __syncwarp();
      }
      ++tcount;
    }
    tc_fence_before();
  } else {
    // ---------------------------------------------------------------- epilogue warps
    const int e = warp - kPersistProducerWarps, q = warp & 3;  // q: the TMEM lane quarter this warp may read
    pg::EpiCtx cx;
    cx.patch = smem_base + kPersistOffPatch + e * pg::kPatchFloats * 4;
    cx.stats = smem_base + kPersistOffStats;
    cx.e = e; cx.lane = lane; cx.et = threadIdx.x - kPersistProducerWarps * 32;
    cx.release_remote = false;
    cx.bn_acc = g.bn.acc;
    cx.bn_H = g.bn.H;
    cx.M = M;
    cx.ldc = g.ldc;
    cx.floor = g.relu ? 0.f : -INFINITY;
    pg::Cursor cur{0, sch.u0};
    pg::Item it;
    uint32_t tcount = 0;
    while (pg::next_item<1>(sch, cur, it)) {
      const uint32_t b = tcount & 1u;
      cx.m_q0 = it.m0 + q * 32;
      cx.n0 = it.n0;
      cx.Cq = g.C + (int64_t)cx.m_q0 * g.ldc + it.n0;
      cx.bias = g.bias ? g.bias + it.n0 : nullptr;
      cx.taddr = tmem_base + ((uint32_t)(q * 32) << 16) + b * BN;
      cx.release_bar = acce0 + 8 * b;
      if (tcount < 8 && q == 0) TRACE(16 + tcount * 8 + 4);
      mbar_wait(accf0 + 8 * b, (tcount >> 1) & 1u);
      tc_fence_after();
      if (tcount < 8 && q == 0) TRACE(16 + tcount * 8 + 5);
      const int m = cx.m_q0 + lane;
      cx.rs = (g.row_scale && m < M) ? __ldg(g.row_scale + m) : 1.f;
      const bool full = cx.m_q0 + 32 <= M;
      if (cx.bn_acc) {
        if (full) pg::epilogue_tile<false, true, true, false, 4>(cx); else pg::epilogue_tile<false, true, false, false, 4>(cx);
      } else {
        if (full) pg::epilogue_tile<false, false, true, false, 4>(cx); else pg::epilogue_tile<false, false, false, false, 4>(cx);
      }
      if (tcount < 8 && q == 0) TRACE(16 + tcount * 8 + 6);
      ++tcount;
    }
  }
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
  // uniform over the grid: every CTA takes a ticket, the last one finalises the statistics
  if (g.bn.acc && last_block_ticket(g.bn.ticket, gridDim.x)) bn_finalize(g.bn, M);
}

}  // namespace tc

#ifdef EIMS_GEMM_TRACE
extern "C" __attribute__((visibility("default"))) int eims_debug_trace_read(unsigned long long* out, int n) {
  if (n > tc::kTraceCtas * tc::kTraceSlots) n = tc::kTraceCtas * tc::kTraceSlots;
  return cudaMemcpyFromSymbol(out, tc::g_trace, (size_t)n * sizeof(unsigned long long)) == cudaSuccess ? 0 : -2;
}
#endif

namespace {

// Tile shape and split-K factor of one problem.  `budget` = CTAs this problem should aim for
// (148 alone, 74 when it shares the launch with a second problem).
int configure(tc::Args& g, int accumulate, int budget, bool* wide_out, bool* need_memset) {
  using namespace tc;
  if (g.M <= 0 || g.N <= 0 || g.K <= 0) return EIMS_ERR_ARG;
  if (g.bn.acc && (accumulate != 0 || g.bn.H != g.N)) return EIMS_ERR_ARG;
  g.vec_a = ((reinterpret_cast<uintptr_t>(g.A) & 15) == 0) && (g.lda % 4 == 0);
  g.vec_b = ((reinterpret_cast<uintptr_t>(g.B) & 15) == 0) && (g.ldb % 4 == 0);
  // 128 x 256 tiles (A read once per row block, 2 stages) when the problem is tall enough to
  // fill the chip with them; 128 x 128 tiles (3 stages) otherwise.
  const bool wide = (g.N % 256 == 0) && ((int64_t)((g.M + BM - 1) / BM) * (g.N / 256) >= 64 || (accumulate == 1 && g.K >= 4096));
  const int BN = wide ? 256 : 128;
  const int mt = (g.M + BM - 1) / BM, nt = (g.N + BN - 1) / BN;
  const int kblocks = (g.K + BK - 1) / BK;
  constexpr int min_kb = 2;  // fewest k-blocks a split-K slice may get
  int splits = 1;
  g.accumulate = accumulate;
  *need_memset = false;
  if (accumulate == 1) {  // split-K: weight gradients reduce over atoms / graphs
    splits = (budget + mt * nt - 1) / (mt * nt);
    const int maxs = (kblocks + min_kb - 1) / min_kb;  // at least min_kb k-blocks per slice
    if (splits > maxs) splits = maxs;
    if (splits < 1) splits = 1;
  } else if (accumulate == 2 || accumulate == 3) {
    // store semantics, but the caller tolerates atomic accumulation order (backward dgrads of the
    // 512-row head): when the tile grid cannot fill the chip, split K and add into a zeroed C.
    g.accumulate = 0;
    if (!g.relu && !g.row_scale && mt * nt <= budget / 4 && kblocks >= 8 && g.ldc == g.N) {
      splits = budget / (mt * nt);
      const int maxs = kblocks / min_kb;
      if (splits > maxs) splits = maxs;
      if (splits > 1) {
        *need_memset = accumulate == 2;  // accumulate == 3: the caller has zeroed C already
        g.accumulate = 1;
      } else {
        splits = 1;
      }
    }
  }
  g.nt = nt; g.mt = mt; g.splits = splits;
  *wide_out = wide;
  return 0;
}

int set_attrs() {
  using namespace tc;
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e1 = cudaFuncSetAttribute(gemm_3xtf32_kernel<128, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 3 * (2 * BM * BK * 4 + 2 * 128 * BK * 4) + 1024);
    cudaError_t e2 = cudaFuncSetAttribute(gemm_3xtf32_kernel<256, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * (2 * BM * BK * 4 + 2 * 256 * BK * 4) + 1024);
    cudaError_t e3 = cudaFuncSetAttribute(gemm_3xtf32_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPersistSmem);
    if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) return EIMS_ERR_CUDA;
    attr_done = true;
  }
  return 0;
}

// The persistent kernel takes a single store problem with >= 4 tiles of 128 x 256 per SM: full 256-wide column tiles,
// vector stores, K <= 512 (single accumulator).  The grouped data-gradient + weight-gradient launch of a GraphConv layer
// stays with one CTA per tile: in this kernel it measured 44.9 us against 40.0 us at BASELINE cfg 2 (B200, stage
// timing), because four epilogue warps share the issue slots with sixteen producer warps that spend ~500 instructions
// per k-block on the hi / lo split.  The planes kernel (gemm_tma.cu), whose producer is one lane driving the copy
// engine, does not have that problem.
bool use_persistent(const tc::Args& g, bool wide) {
  using namespace tc;
  if (!wide || g.accumulate) return false;
  if ((g.N % 256) || (g.ldc & 3) || (reinterpret_cast<uintptr_t>(g.C) & 15)) return false;
  if (g.bias && (reinterpret_cast<uintptr_t>(g.bias) & 15)) return false;
  if ((g.K + BK - 1) / BK > pg::kMaxKbPerItem) return false;   // upper bound when K lives on the device (capacity)
  if ((int64_t)g.mt * g.nt * ((g.K + BK - 1) / BK) * 148 > (int64_t)1 << 30) return false;  // 32-bit schedule arithmetic
  return g.mt * g.nt >= 4 * 148;
}

int launch_group(const tc::Group& grp_in, int ctas, bool wide, cudaStream_t st, int nprob) {
  using namespace tc;
  const int BN = wide ? 256 : 128, stages = wide ? 2 : 3;
  const int smem_bytes = stages * (2 * BM * BK * 4 + 2 * BN * BK * 4) + 1024;
  cudaError_t e;
  if (nprob == 1 && use_persistent(grp_in.g[0], wide)) {
    e = launch_pdl(gemm_3xtf32_persistent_kernel, dim3(148), dim3(kPersistThreads), kPersistSmem, st, grp_in.g[0]);
  } else {
    e = wide ? launch_pdl(gemm_3xtf32_kernel<256, 2>, dim3(ctas), dim3(kThreads), smem_bytes, st, grp_in)
             : launch_pdl(gemm_3xtf32_kernel<128, 3>, dim3(ctas), dim3(kThreads), smem_bytes, st, grp_in);
  }
  return e == cudaSuccess ? 0 : EIMS_ERR_CUDA;
}

tc::Args make_args(const GemmProblem& q) {
  tc::Args g{q.A, q.B, q.C, q.lda, q.ldb, q.ldc, q.a_mn, q.b_mn, q.M, q.N, q.K, q.m_dev, q.k_dev, q.row_scale, q.bias,
             q.relu, q.accumulate, 0, 0, dims_early_ref(), 1, 1, 1, BnFuse{}};
  if (q.bn) g.bn = *q.bn;
  return g;
}

}  // namespace

int launch_gemm_tc(const float* A, int lda, int a_mn, const float* B, int ldb, int b_mn, float* C, int ldc, int M,
                   int N, int K, const int* m_dev, const int* k_dev, const float* row_scale, const float* bias,
                   int relu, int accumulate, cudaStream_t st, const BnFuse* bn) {
  GemmProblem q{A, lda, a_mn, B, ldb, b_mn, C, ldc, M, N, K, m_dev, k_dev, row_scale, bias, relu, accumulate, bn};
  tc::Group grp{};
  grp.g[0] = make_args(q);
  bool wide = false, zero = false;
  if (int rc = configure(grp.g[0], accumulate, 148, &wide, &zero)) return rc;
  if (int rc = set_attrs()) return rc;
  if (zero && cudaMemsetAsync(C, 0, (size_t)M * ldc * sizeof(float), st) != cudaSuccess) return EIMS_ERR_CUDA;
  grp.g[1] = grp.g[0];
  grp.ctas0 = grp.g[0].nt * grp.g[0].mt * grp.g[0].splits;
  return launch_group(grp, grp.ctas0, wide, st, 1);
}

// Two independent problems in one launch (the weight gradient and the data gradient of a layer):
// one launch latency and one pipeline fill / drain instead of two, and the second problem's CTAs
// fill the SMs the first leaves idle.  Falls back to two launches when the tile shapes differ.
int launch_gemm_tc_pair(const GemmProblem& p0, const GemmProblem& p1, cudaStream_t st) {
  tc::Group grp{};
  grp.g[0] = make_args(p0);
  grp.g[1] = make_args(p1);
  bool w0 = false, w1 = false, z0 = false, z1 = false;
  if (int rc = configure(grp.g[0], p0.accumulate, 148, &w0, &z0)) return rc;
  if (int rc = configure(grp.g[1], p1.accumulate, 148, &w1, &z1)) return rc;
  if (w0 != w1 || z0 || z1 || p0.bn || p1.bn) {
    if (int rc = launch_gemm_tc(p0.A, p0.lda, p0.a_mn, p0.B, p0.ldb, p0.b_mn, p0.C, p0.ldc, p0.M, p0.N, p0.K, p0.m_dev, p0.k_dev,
                                p0.row_scale, p0.bias, p0.relu, p0.accumulate, st, p0.bn)) return rc;
    return launch_gemm_tc(p1.A, p1.lda, p1.a_mn, p1.B, p1.ldb, p1.b_mn, p1.C, p1.ldc, p1.M, p1.N, p1.K, p1.m_dev, p1.k_dev,
                          p1.row_scale, p1.bias, p1.relu, p1.accumulate, st, p1.bn);
  }
  // small problems share one wave: aim each at half the chip
  const int c0 = grp.g[0].nt * grp.g[0].mt * grp.g[0].splits, c1 = grp.g[1].nt * grp.g[1].mt * grp.g[1].splits;
  if (c0 + c1 > 148 && c0 <= 148 && c1 <= 148 && grp.g[0].nt * grp.g[0].mt <= 37 && grp.g[1].nt * grp.g[1].mt <= 37) {
    if (int rc = configure(grp.g[0], p0.accumulate, 74, &w0, &z0)) return rc;
    if (int rc = configure(grp.g[1], p1.accumulate, 74, &w1, &z1)) return rc;
    if (z0 || z1) return EIMS_ERR_ARG;
  }
  if (int rc = set_attrs()) return rc;
  grp.ctas0 = grp.g[0].nt * grp.g[0].mt * grp.g[0].splits;
  const int ctas = grp.ctas0 + grp.g[1].nt * grp.g[1].mt * grp.g[1].splits;
  return launch_group(grp, ctas, w0, st, 2);
}

}  // namespace eims

EIMS_TIMELINE_READER(gemm_tc)
