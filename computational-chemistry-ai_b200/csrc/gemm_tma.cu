// K3/K6 on PRE-SPLIT operand planes, fed by the tensor-map copy engine (TMA), persistent.
//
// The 3xTF32 product  A*B ~= A_lo*B_hi + A_hi*B_lo + A_hi*B_hi  needs  hi = rna_tf32(x), lo = rna_tf32(x - hi)  of every
// operand element.  gemm_tc.cu computes the split inside the GEMM: 16 producer warps pull fp32 tiles through the
// load/store unit, split them in registers and st.shared them into the UMMA layout - and that load/store + shared-memory
// pipe, not the tensor core, bounds its main loop and leaves no room to overlap an epilogue.  Here the split is done ONCE
// by whoever produces the operand (the aggregation kernel for a_l, the BatchNorm-backward pass for q, a tiny kernel for
// the weights): each operand lives in global memory as two stacked fp32 planes [2][rows][ld] holding tf32-exact values,
// and a k-block of both planes travels global -> shared by ONE cp.async.bulk.tensor (3-D box: k x rows x plane) straight
// into the swizzled layout tcgen05.mma reads:
//     K-major operand  (memory [mn][k]):  box {32 k, ROWS mn, 2}  CU_TENSOR_MAP_SWIZZLE_128B            -> SWIZZLE_128B
//     MN-major operand (memory [k][mn]):  box {32 mn, 32 k, 2}    CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B   -> SWIZZLE_128B_BASE32B
//                                         (one box per 32-wide mn atom, hi and lo of an atom adjacent: LBO = 8 KB)
// A CTA pair per two SMs (192 threads each): warp 0 = copy-engine producer (one lane), warp 1 = MMA issuer (one lane of
// the leader CTA, owns TMEM), warps 2-5 = epilogue.  The pair walks over a list of work items - output tiles of a "store" problem (forward / data
// gradient: 128 x 256 tile, whole K) and k-slices of a "split-K" problem (weight gradient over the atoms: red.global.add)
// - with two 256-column accumulators in TMEM, so the epilogue of item i (TMEM -> registers -> padded shared patch ->
// 128-byte row segments) runs under the main loop of item i+1 and uses nothing the main loop needs.  The items of a
// launch are dealt out on the device from the LIVE sizes (atoms in the batch): store tiles round-robin, then the k-blocks
// of the split-K problem in contiguous ranges sized so that every CTA ends at the same time.
#include <cuda.h>

#include <cstring>

#include "common.cuh"
#include "gemm_persist.cuh"
#include "launchers.h"

namespace eims {

namespace tma {

// Optional pipeline trace (-DEIMS_GEMM_TRACE, tools/gemm_planes_trace.py): SM-clock stamps of the roles of a few CTAs.
#ifdef EIMS_GEMM_TRACE
constexpr int kTraceCtas = 8, kTraceSlots = 64;
__device__ unsigned long long g_ptrace[kTraceCtas * kTraceSlots];
#define PTRACE(slot)                                                                          \
  do {                                                                                        \
    const int _c = blockIdx.x;                                                                \
    if (_c < kTraceCtas && (threadIdx.x & 31) == 0 && (slot) < kTraceSlots) g_ptrace[_c * kTraceSlots + (slot)] = clock64(); \
  } while (0)
#else
#define PTRACE(slot) do { } while (0)
#endif

using namespace pg;   // tile constants, work-item schedule and tile epilogue shared with gemm_tc.cu (gemm_persist.cuh)
constexpr int kThreads = (2 + kEpiWarps) * 32;
constexpr int kMaxKbDeep = 64;                                     // "deep" launches (main + correction accumulator): K <= 2048
// A CTA pair (cluster of two SMs) works on a 256 x 256 tile with tcgen05.mma.cta_group::2 - each CTA stages its own
// 128 rows of A and HALF of B (128 of the 256 columns), the tensor cores of both SMs read both halves: per CTA and
// k-block 64 KB instead of 96 KB enter shared memory and 96 KB instead of 144 KB are read back by the MMAs, which takes
// the main loop from shared-memory-bandwidth-bound (240 KB / 128 B per clock = 1.9 k cycles per k-block, measured with
// one CTA per 128 x 256 tile) to MMA-issue-bound (1.54 k), and the smaller stage buys a third stage.
constexpr int PAIR = 2;
constexpr int STAGES = 3;
constexpr int B_ROWS = BN / PAIR;
static_assert(B_ROWS == kTmaBRows, "the B maps are encoded with a box of kTmaBRows rows");
constexpr int A_PLANE = BM * BK * 4, B_PLANE = B_ROWS * BK * 4;   // 16 KB each
constexpr int STAGE_BYTES = 2 * A_PLANE + 2 * B_PLANE;            // A hi, A lo, B hi, B lo: 64 KB
constexpr int OFF_PATCH = STAGES * STAGE_BYTES;
constexpr int OFF_STATS = OFF_PATCH + kEpiWarps * kPatchFloats * 4;
constexpr int OFF_BARS = OFF_STATS + kEpiWarps * 2 * kStatCols * 8;
constexpr int OFF_MISC = OFF_BARS + 16 * 8;                      // full[S], empty[S], acc_full[2], acc_empty[2]
constexpr int kSmemBytes = OFF_MISC + 64 + 1024;                 // + slack for the 1024-byte round-up of the base

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
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
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tma_prefetch_desc(const void* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// UMMA shared-memory matrix descriptor (sm_100 format): see gemm_tc.cu
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)layout_type << 61;
  return d;
}

struct Prob {
  CUtensorMap ta, tb;                  // stacked hi / lo planes of A and of B
  float* C;
  int ldc, a_mn, b_mn;
  int M, N, K;                         // static sizes (capacities where a live size exists)
  const int* m_dev; const int* k_dev;  // live sizes on the device (atoms in the batch) or null
  const float* row_scale; const float* bias;
  int relu, red;                       // red != 0: split-K problem, partial sums added with red.global.add
  BnFuse bn;                           // bn.acc != null: column sums of the stored tile -> BatchNorm statistics
};
struct Group {
  Prob g[2];
  int nprob, early, ovh;               // ovh: fixed cost of one item in k-block units (balances the two problems)
  // deep != 0 (a store problem with K > 512): every item of the launch uses BOTH 256-column accumulators - the A_hi*B_hi
  // products in one, the two correction products in the other, summed in the epilogue - because the tensor core truncates
  // on every accumulation and one accumulator over K = 1024 carries a bias of ~1e-5 (gemm_tc.cu, measured); the epilogue
  // of an item then no longer overlaps the next item's main loop, which at >= 32 k-blocks per item costs ~10 %.
  int deep;
};

// ---- CTA-pair plumbing
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t mapa_rank(uint32_t addr, uint32_t rank) {   // shared::cluster address of `addr` in CTA `rank`
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// 3-D tiled tensor-map load (coordinates innermost first), issued by either CTA of a pair: completion bytes go to the
// LEADER's mbarrier (shared::cluster address)
__device__ __forceinline__ void tma_load_3d_pair(uint32_t dst, const void* map, int c0, int c1, int c2, uint32_t leader_bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(leader_bar)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_tf32_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {   // arrives on `bar` in BOTH CTAs of the pair
  const uint16_t mask = 3;
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(mask) : "memory");
}

__global__ void __launch_bounds__(kThreads, 1) gemm_planes_kernel(const __grid_constant__ Group grp) {
  constexpr int S = STAGES;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BARS);   // full[S], empty[S], acc_full[2], acc_empty[2]
  uint32_t* misc = reinterpret_cast<uint32_t*>(smem + OFF_MISC);   // [0] TMEM base
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0) PTRACE(0);
  const uint32_t rank = cluster_ctarank();                            // rank 0 of a pair issues the MMAs
  const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[S]), accf0 = smem_u32(&bars[2 * S]), acce0 = smem_u32(&bars[2 * S + 2]);
  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(full0 + 8 * s, 1);
      mbar_init(empty0 + 8 * s, 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(accf0 + 8 * s, 1);
      mbar_init(acce0 + 8 * s, kEpiWarps * PAIR);   // the leader's copy also counts the peer's epilogue warps
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    for (int k = 0; k < grp.nprob; ++k) { tma_prefetch_desc(&grp.g[k].ta); tma_prefetch_desc(&grp.g[k].tb); }
  }
  if (warp == 1) tmem_alloc_pair(smem_u32(&misc[0]), 512);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // the peer's barriers are initialised before anything remote touches them
  tc_fence_after();
  const uint32_t tmem_base = misc[0];
  const uint32_t smem_base = smem_u32(smem);
  int Mv[2], Kv[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    Mv[k] = grp.g[k].M; Kv[k] = grp.g[k].K;
    if (grp.early && k < grp.nprob) {
      if (grp.g[k].m_dev) Mv[k] = __ldcg(grp.g[k].m_dev);
      if (grp.g[k].k_dev) Kv[k] = __ldcg(grp.g[k].k_dev);
    }
  }
  if (warp == 0) PTRACE(1);
  pdl_sync();
  if (warp == 0) PTRACE(2);
  if (!grp.early) {
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      if (k < grp.nprob) {
        if (grp.g[k].m_dev) Mv[k] = __ldcg(grp.g[k].m_dev);
        if (grp.g[k].k_dev) Kv[k] = __ldcg(grp.g[k].k_dev);
      }
    }
  }
  SchedIn sin;
  sin.nprob = grp.nprob; sin.ovh = grp.ovh;
  sin.red[0] = grp.g[0].red; sin.red[1] = grp.g[1].red; sin.N[0] = grp.g[0].N; sin.N[1] = grp.g[1].N;
  const Sched sch = make_sched<PAIR>(sin, Mv, Kv);

  if (warp == 0) {
    // ---------------------------------------------------------------- copy-engine producer (every CTA: its rows of A, its part of B)
    if (lane == 0) {
      Cursor cur{0, sch.u0};
      Item it;
      uint32_t n = 0, tcount = 0;
      while (next_item<PAIR>(sch, cur, it)) {
        // (fields of the selected problem go into registers once per item: an indexed read of the kernel-parameter
        // bank inside the loops below costs ~100 cycles each time)
        const int pi = it.prob;
        const void* const map_a = pi ? (const void*)&grp.g[1].ta : (const void*)&grp.g[0].ta;
        const void* const map_b = pi ? (const void*)&grp.g[1].tb : (const void*)&grp.g[0].tb;
        const int a_mn = pi ? grp.g[1].a_mn : grp.g[0].a_mn, b_mn = pi ? grp.g[1].b_mn : grp.g[0].b_mn;
        const int m_own = it.m0 + (int)rank * BM, n_own = it.n0 + (int)rank * B_ROWS;
        PTRACE(8 + tcount * 8 + 0);   // first copy of the item about to be issued
        ++tcount;
        for (int i = 0; i < it.nkb; ++i, ++n) {
          const uint32_t s = n % S;
          mbar_wait(empty0 + 8 * s, ((n / S) & 1u) ^ 1u);
          uint32_t bar = full0 + 8 * s;
          if (rank == 0) mbar_expect_tx(bar, STAGE_BYTES * PAIR);
          bar = mapa_rank(bar, 0);
          const uint32_t sa = smem_base + s * STAGE_BYTES, sb = sa + 2 * A_PLANE;
          const int k0 = (it.kb0 + i) * BK;
          if (!a_mn) {
            tma_load_3d_pair(sa, map_a, k0, m_own, 0, bar);
          } else {
#pragma unroll
            for (int j = 0; j < BM / 32; ++j) tma_load_3d_pair(sa + j * 8192, map_a, m_own + 32 * j, k0, 0, bar);
          }
          if (!b_mn) {
            tma_load_3d_pair(sb, map_b, k0, n_own, 0, bar);
          } else {
#pragma unroll
            for (int j = 0; j < B_ROWS / 32; ++j) tma_load_3d_pair(sb + j * 8192, map_b, n_own + 32 * j, k0, 0, bar);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ---------------------------------------------------------------- MMA issuer (the leader CTA of a pair only)
    if (rank == 0) {
      Cursor cur{0, sch.u0};
      Item it;
      uint32_t n = 0, tcount = 0;
      while (next_item<PAIR>(sch, cur, it)) {
        const int a_mn = it.prob ? grp.g[1].a_mn : grp.g[0].a_mn, b_mn = it.prob ? grp.g[1].b_mn : grp.g[0].b_mn;
        const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
                               ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((BM * PAIR) >> 4) << 24);
        // K-major: rows of 128 bytes, 8-row groups 1024 B apart (SBO), k-step (8 tf32) = +32 B, lo plane after the hi plane.
        // MN-major: per 32-wide mn atom one 8 KB box = hi (32 k-rows x 128 B) then lo; LBO = 8192 (next atom),
        //           SBO = 512 (next 4 k-rows), k-step (8 k-rows) = +1024 B, lo = hi + 4096.
        const uint32_t a_lbo = a_mn ? 8192u : 16u, a_sbo = a_mn ? 512u : 1024u, a_kstep = a_mn ? 1024u : 32u;
        const uint32_t b_lbo = b_mn ? 8192u : 16u, b_sbo = b_mn ? 512u : 1024u, b_kstep = b_mn ? 1024u : 32u;
        const uint32_t a_lo_off = a_mn ? 4096u : (uint32_t)A_PLANE, b_lo_off = b_mn ? 4096u : (uint32_t)B_PLANE;
        const uint32_t a_lt = a_mn ? 1u : 2u, b_lt = b_mn ? 1u : 2u;
        const uint32_t b = grp.deep ? 0u : (tcount & 1u);
        const uint32_t bph = grp.deep ? (tcount & 1u) : ((tcount >> 1) & 1u);
        mbar_wait(acce0 + 8 * b, bph ^ 1u);  // accumulator b drained by the epilogue warps (of both CTAs)
        tc_fence_after();
        PTRACE(8 + tcount * 8 + 1);   // accumulator free
        const uint32_t acc = tmem_base + b * BN;
        const uint32_t acc_corr = grp.deep ? tmem_base + BN : acc;   // deep: the correction products have their own accumulator
        for (int i = 0; i < it.nkb; ++i, ++n) {
          const uint32_t s = n % S;
          mbar_wait(full0 + 8 * s, (n / S) & 1u);
          tc_fence_after();
          if (i == 0) PTRACE(8 + tcount * 8 + 2);              // first k-block landed
          if (i == it.nkb - 1) PTRACE(8 + tcount * 8 + 3);     // last k-block landed
          if (lane == 0) {
            const uint32_t sa = smem_base + s * STAGE_BYTES, sb = sa + 2 * A_PLANE;
#pragma unroll
            for (int ks = 0; ks < BK / 8; ++ks) {
              const uint64_t dah = make_desc(sa + ks * a_kstep, a_lbo, a_sbo, a_lt);
              const uint64_t dal = make_desc(sa + a_lo_off + ks * a_kstep, a_lbo, a_sbo, a_lt);
              const uint64_t dbh = make_desc(sb + ks * b_kstep, b_lbo, b_sbo, b_lt);
              const uint64_t dbl = make_desc(sb + b_lo_off + ks * b_kstep, b_lbo, b_sbo, b_lt);
              const uint32_t first = (i > 0 || ks > 0) ? 1u : 0u;
              const uint32_t mfirst = grp.deep ? first : 1u;   // deep: the main accumulator starts with this product
              umma_tf32_pair(acc_corr, dal, dbh, idesc, first);  // smallest terms first
              umma_tf32_pair(acc_corr, dah, dbl, idesc, 1u);
              umma_tf32_pair(acc, dah, dbh, idesc, mfirst);
            }
            umma_commit_pair(empty0 + 8 * s);                        // frees the stage in both CTAs when these MMAs retire
            if (i == it.nkb - 1) umma_commit_pair(accf0 + 8 * b);    // accumulator b complete (both halves)
          }
          __syncwarp();
        }
        ++tcount;
      }
      tc_fence_before();
    }
  } else {
    // ---------------------------------------------------------------- epilogue warps (each CTA drains its own 128 rows)
    const int e = warp - 2, q = warp & 3;  // q: the TMEM lane quarter this warp may read
    EpiCtx cx;
    cx.patch = smem_base + OFF_PATCH + e * kPatchFloats * 4;   // shared-space byte addresses
    cx.stats = smem_base + OFF_STATS;                             // double [kEpiWarps][2][kStatCols]
    cx.e = e; cx.lane = lane; cx.et = threadIdx.x - 64;
    Cursor cur{0, sch.u0};
    Item it;
    uint32_t tcount = 0;
    while (next_item<PAIR>(sch, cur, it)) {
      // the selected problem's fields in registers (an indexed read of the kernel-parameter bank costs ~100 cycles)
      const bool p1 = it.prob != 0;
      const float* const row_scale = p1 ? grp.g[1].row_scale : grp.g[0].row_scale;
      const float* const bias = p1 ? grp.g[1].bias : grp.g[0].bias;
      const bool relu = (p1 ? grp.g[1].relu : grp.g[0].relu) != 0, red = (p1 ? grp.g[1].red : grp.g[0].red) != 0;
      cx.bn_acc = p1 ? grp.g[1].bn.acc : grp.g[0].bn.acc;
      cx.bn_H = p1 ? grp.g[1].bn.H : grp.g[0].bn.H;
      const int ldc = p1 ? grp.g[1].ldc : grp.g[0].ldc;
      const int M = p1 ? Mv[1] : Mv[0];
      const int m_own = it.m0 + (int)rank * BM;
      const uint32_t b = grp.deep ? 0u : (tcount & 1u);
      const uint32_t bph = grp.deep ? (tcount & 1u) : ((tcount >> 1) & 1u);
      cx.m_q0 = m_own + q * 32;
      cx.M = M;
      cx.n0 = it.n0;
      cx.ldc = ldc;
      cx.Cq = (p1 ? grp.g[1].C : grp.g[0].C) + (int64_t)cx.m_q0 * ldc + it.n0;
      cx.bias = (bias && (!red || it.kb0 == 0)) ? bias + it.n0 : nullptr;
      cx.floor = relu ? 0.f : -INFINITY;
      cx.taddr = tmem_base + ((uint32_t)(q * 32) << 16) + b * BN;
      // what hands accumulator b back to the MMA issuer (the leader's barrier also counts the peer's warps)
      cx.release_bar = rank != 0 ? mapa_rank(acce0 + 8 * b, 0) : acce0 + 8 * b;
      cx.release_remote = rank != 0;
      if (e == 0) PTRACE(8 + tcount * 8 + 4);                  // epilogue waits for the accumulator
      mbar_wait(accf0 + 8 * b, bph);
      tc_fence_after();
      if (e == 0) PTRACE(8 + tcount * 8 + 5);                  // accumulator complete
      const int m = cx.m_q0 + lane;
      cx.rs = (row_scale && m < M) ? __ldg(row_scale + m) : 1.f;
      const bool full = cx.m_q0 + 32 <= M;
      if (grp.deep) {   // (the guarded variants only: a deep launch is MMA-bound, the epilogue is a few per cent of it)
        if (red) epilogue_tile<true, false, false, true>(cx);
        else if (cx.bn_acc) epilogue_tile<false, true, false, true>(cx);
        else epilogue_tile<false, false, false, true>(cx);
      } else if (red) {
        if (full) epilogue_tile<true, false, true, false>(cx); else epilogue_tile<true, false, false, false>(cx);
      } else if (cx.bn_acc) {
        if (full) epilogue_tile<false, true, true, false>(cx); else epilogue_tile<false, true, false, false>(cx);
      } else {
        if (full) epilogue_tile<false, false, true, false>(cx); else epilogue_tile<false, false, false, false>(cx);
      }
      if (e == 0) PTRACE(8 + tcount * 8 + 6);                  // tile stored
      ++tcount;
    }
  }
  if (warp == 0) PTRACE(3);
  __syncthreads();
  cluster_sync_all();   // nothing remote (barrier arrivals, the peer's MMA reads of this CTA's tiles) is still in flight
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, 512);
  }
  for (int k = 0; k < grp.nprob; ++k) {
    if (grp.g[k].bn.acc) {  // uniform over the grid: every CTA takes a ticket, the last one finalises the statistics
      if (last_block_ticket(grp.g[k].bn.ticket, gridDim.x)) bn_finalize(grp.g[k].bn, Mv[k]);
    }
  }
  if (warp == 0) PTRACE(4);
}

// x -> (hi, lo) planes, elementwise:  hi = rna_tf32(x), lo = rna_tf32(x - hi)   (the split of gemm_tc.cu)
__global__ void __launch_bounds__(256) split_planes_kernel(const float4* __restrict__ src, float4* __restrict__ hi,
                                                           float4* __restrict__ lo, int64_t n4, int wait) {
  if (wait) pdl_sync();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 v = __ldg(src + i);
    float4 h, l;
    split_tf32_planes(v.x, h.x, l.x); split_tf32_planes(v.y, h.y, l.y);
    split_tf32_planes(v.z, h.z, l.z); split_tf32_planes(v.w, h.w, l.w);
    hi[i] = h;
    lo[i] = l;
  }
}

}  // namespace tma

#ifdef EIMS_GEMM_TRACE
extern "C" __attribute__((visibility("default"))) int eims_debug_trace_read_planes(unsigned long long* out, int n) {
  if (n > tma::kTraceCtas * tma::kTraceSlots) n = tma::kTraceCtas * tma::kTraceSlots;
  if (cudaMemcpyFromSymbol(out, tma::g_ptrace, (size_t)n * sizeof(unsigned long long)) != cudaSuccess) return -2;
  static unsigned long long zeros[tma::kTraceCtas * tma::kTraceSlots];
  return cudaMemcpyToSymbol(tma::g_ptrace, zeros, sizeof(zeros)) == cudaSuccess ? 0 : -2;
}
#endif

namespace {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
    else
      cudaGetLastError();
  }
  return fn;
}

}  // namespace

static_assert(sizeof(TmaMap) == sizeof(CUtensorMap), "TmaMap must mirror CUtensorMap");

// Tensor map over the stacked planes [2][rows][ld] of a row-major operand with `cols` live columns.
//   mn_major = 0: the rows are the operand's M / N index and the columns its K index; box {32 k, box_rows, 2}
//   mn_major = 1: the rows are the K index and the columns the M / N index;            box {32 mn, 32 k, 2}
int tma_make_map(TmaMap* out, const float* planes, int64_t plane_stride, int rows, int cols, int ld, int box_rows, int mn_major) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return EIMS_ERR_CUDA;
  if (!out || !planes || rows < 1 || cols < 32 || (ld & 3) || (plane_stride & 3) || (reinterpret_cast<uintptr_t>(planes) & 15))
    return EIMS_ERR_ARG;
  if (!mn_major && (box_rows < 8 || box_rows > 256)) return EIMS_ERR_ARG;
  cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, 2};
  cuuint64_t strides[2] = {(cuuint64_t)ld * 4, (cuuint64_t)plane_stride * 4};
  cuuint32_t box[3] = {32, (cuuint32_t)(mn_major ? 32 : box_rows), 2};
  cuuint32_t estr[3] = {1, 1, 1};
  CUtensorMap m;
  const CUresult r = fn(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(planes), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return EIMS_ERR_CUDA;
  memcpy(out, &m, sizeof(m));
  return 0;
}

bool gemm_tma_enabled() { return encode_fn() != nullptr; }

// shapes the planes kernel takes: full 256-wide column tiles, vector stores, K of a store problem <= 2048 (> 512: deep mode)
bool gemm_tma_supports(const GemmTmaProblem& q) {
  if (q.N < 256 || (q.N % 256) || (q.ldc & 3) || (reinterpret_cast<uintptr_t>(q.C) & 15)) return false;
  if (q.bias && (reinterpret_cast<uintptr_t>(q.bias) & 15)) return false;
  if (!q.red && (q.K + 31) / 32 > tma::kMaxKbDeep) return false;
  if (q.bn && (q.red || q.bn->H != q.N)) return false;
  return q.M > 0 && q.K > 0 && q.ta && q.tb;
}

int launch_gemm_tma(const GemmTmaProblem* p0, const GemmTmaProblem* p1, cudaStream_t st) {
  using namespace tma;
  if (!p0 || !gemm_tma_supports(*p0) || (p1 && !gemm_tma_supports(*p1))) return EIMS_ERR_ARG;
  if (p1 && (p0->red != 0) == (p1->red != 0)) return EIMS_ERR_ARG;  // one store problem and one split-K problem at most
  static bool attr_done = false;
  if (!attr_done) {
    if (cudaFuncSetAttribute(gemm_planes_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes) != cudaSuccess)
      return EIMS_ERR_CUDA;
    attr_done = true;
  }
  constexpr int kItemOverhead = 4;  // fixed cost of one work item in k-block units (balances the two problems)
  Group grp;
  memset(&grp, 0, sizeof(grp));
  const GemmTmaProblem* ps[2] = {p0, p1};
  int64_t items = 0;
  for (int k = 0; k < 2; ++k) {
    const GemmTmaProblem* q = ps[k] ? ps[k] : p0;
    Prob& g = grp.g[k];
    memcpy(&g.ta, q->ta, sizeof(CUtensorMap));
    memcpy(&g.tb, q->tb, sizeof(CUtensorMap));
    g.C = q->C; g.ldc = q->ldc; g.a_mn = q->a_mn; g.b_mn = q->b_mn;
    g.M = q->M; g.N = q->N; g.K = q->K; g.m_dev = q->m_dev; g.k_dev = q->k_dev;
    g.row_scale = q->row_scale; g.bias = q->bias; g.relu = q->relu; g.red = q->red;
    if (q->bn) g.bn = *q->bn;
    if (ps[k]) items += (int64_t)((q->M + BM * PAIR - 1) / (BM * PAIR)) * (q->N / BN) * (q->red ? 148 : 1);
    // the device-side schedule works in 32-bit integers (k-block units times CTAs)
    if (ps[k] && (int64_t)((q->M + BM - 1) / BM) * (q->N / BN) * ((q->K + BK - 1) / BK) * 148 >= ((int64_t)1 << 31)) return EIMS_ERR_ARG;
  }
  grp.nprob = p1 ? 2 : 1;
  for (int k = 0; k < grp.nprob; ++k)
    if (!grp.g[k].red && (grp.g[k].K + 31) / 32 > kMaxKbPerItem) grp.deep = 1;
  grp.early = dims_early_ref();
  grp.ovh = kItemOverhead;
  const int units = 148 / PAIR;
  int grid = (int)(items < units ? items : units) * PAIR;
  if (grid < PAIR) grid = PAIR;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  attr[1].id = cudaLaunchAttributeClusterDimension;
  attr[1].val.clusterDim.x = PAIR;
  attr[1].val.clusterDim.y = 1;
  attr[1].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  cudaError_t e = cudaLaunchKernelEx(&cfg, gemm_planes_kernel, grp);
  return e == cudaSuccess ? 0 : EIMS_ERR_CUDA;
}

int launch_split_planes(const float* src, float* hi, float* lo, int64_t n, cudaStream_t st, bool chained) {
  if ((n & 3) || ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(hi) | reinterpret_cast<uintptr_t>(lo)) & 15)) return EIMS_ERR_ARG;
  const int64_t n4 = n / 4;
  int blocks = (int)((n4 + 255) / 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  cudaError_t e;
  if (chained) e = launch_pdl(tma::split_planes_kernel, dim3(blocks), dim3(256), 0, st, reinterpret_cast<const float4*>(src),
                              reinterpret_cast<float4*>(hi), reinterpret_cast<float4*>(lo), n4, 1);
  else {
    tma::split_planes_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<const float4*>(src), reinterpret_cast<float4*>(hi),
                                                    reinterpret_cast<float4*>(lo), n4, 0);
    e = cudaGetLastError();
  }
  return e == cudaSuccess ? 0 : EIMS_ERR_CUDA;
}

}  // namespace eims

EIMS_TIMELINE_READER(gemm_tma)
