// Data-parallel optimiser step in ONE kernel: gradient all-reduce + AdamW + parameter broadcast
// over NVLink / NVSwitch peer memory (new functionality - the reference is single-GPU, GCN:63;
// semantics = PyTorch DDP mean of per-rank gradients followed by GCN:429 `optimizer.step()`).
//
//   every rank r owns the slice [r*per, (r+1)*per) of the flat parameter vector
//   phase 0  cross-GPU barrier "gradients of this step are complete everywhere"
//   phase 1  g   = sum over ranks of grads[slice]       multimem.ld_reduce (the NVSwitch adds, one
//                                                       reduced stream comes back) or peer loads
//            AdamW on the slice (m, v exist for the own slice only - ZeRO-1 style)
//            p  -> every rank's parameter buffer        multimem.st (switch multicast) or peer stores
//            the gradient buffer of the PREVIOUS step (double-buffered) is zeroed for reuse
//   phase 2  cross-GPU barrier "all slices of the new parameters have landed here"
// Per rank and step the links carry ~P*4 bytes in and out (3.15 MB at BASELINE cfg 2-4) instead
// of an NCCL all-reduce followed by a separate AdamW launch; every rank ends with bit-identical
// parameters because each element is updated by exactly one rank.
//
// Barriers are monotonically increasing sequence numbers in each rank's signal pad
// (st.release.sys / ld.acquire.sys); ranks are different GPUs, so spinning is safe.
#include "common.cuh"
#include "launchers.h"

namespace eims {

constexpr int kMaxRanks = 16;

struct DpPeers {
  float* grads[kMaxRanks];       // this step's gradient buffer of every rank (peer-mapped)
  float* params[kMaxRanks];      // parameter buffer of every rank (peer-mapped)
  uint32_t* signals[kMaxRanks];  // signal pad of every rank: [2][kMaxRanks] words used
  float* grads_mc;               // multicast (NVLS) address of the gradient buffers, or null
  float* params_mc;              // multicast address of the parameter buffers, or null
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float4 multimem_ld_reduce_add(const float* mc) {
  float4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(mc)
               : "memory");
  return v;
}
__device__ __forceinline__ void multimem_st(float* mc, float4 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w)
               : "memory");
}

// Wait until every rank has written `seq` (or later) into this rank's pad row `row`.  A peer may be late for a
// long time for honest reasons (rank 0 writing a checkpoint or running the eval pass, an I/O stall, lazy module
// loading on the first step), so the wait is long (EIMS_DP_TIMEOUT_S, default 600 s, measured on %globaltimer)
// and running out of it is reported, not trapped: the waiting thread records the sequence number in `*status`
// (read by the host with the per-epoch flag check) and the kernel carries on, so the context survives and the
// job can stop with an error message instead of a sticky CUDA fault on every rank.
__device__ __forceinline__ void wait_all(const uint32_t* my_pad, int row, int world, uint32_t seq, unsigned long long timeout_ns,
                                         uint32_t* status) {
  if ((int)threadIdx.x < world) {
    const uint32_t* p = my_pad + row * kMaxRanks + threadIdx.x;
    unsigned long long t0 = 0;
    unsigned int spins = 0;
    while ((int32_t)(ld_acquire_sys(p) - seq) < 0) {
      if ((++spins & 0x3ffu) == 0) {  // look at the clock every 1024 polls
        unsigned long long now;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        if (t0 == 0) t0 = now;
        else if (now - t0 > timeout_ns) { atomicMax(status, seq ? seq : 1u); break; }
      }
    }
  }
  __syncthreads();
}

// The kernel works on the range [base4, base4 + n4) (in float4 units) of the flat buffers, so a step
// can exchange the head bucket early (on a side stream, while the GCN layers are still being
// differentiated) and the GCN / BatchNorm bucket at the end; `row` selects the bucket's pair of
// signal rows.
__global__ void __launch_bounds__(256) dp_adamw_kernel(DpPeers pr, int rank, int world, float* __restrict__ m,
                                                       float* __restrict__ v, float* __restrict__ zero_buf,
                                                       int64_t base4, int64_t n4, int64_t per, uint32_t seq, int row,
                                                       unsigned int* ticket, AdamK k, const StepBlock* __restrict__ blk,
                                                       unsigned long long timeout_ns) {
  pdl_sync();
  if (blk) { k = blk->adam; seq = blk->dp_seq; }  // captured graph: this step's scalars / sequence number
  uint32_t* status = ticket + 1;
  uint32_t* my_pad = pr.signals[rank];
  // ---- phase 0: my gradients are complete (stream order) -> tell everyone, wait for everyone
  if (blockIdx.x == 0 && (int)threadIdx.x < world) {
    __threadfence_system();
    st_release_sys(pr.signals[threadIdx.x] + (2 * row) * kMaxRanks + rank, seq);
  }
  wait_all(my_pad, 2 * row, world, seq, timeout_ns, status);
  // ---- phase 1: reduce + AdamW + broadcast of the own slice
  const int64_t s0 = base4 + (int64_t)rank * per, s1 = min(base4 + n4, s0 + per);
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
  // kDpUnroll independent reductions in flight per thread: a multimem.ld_reduce is a round trip through the
  // switch (microseconds), and at 2 GPUs a thread owns 2-3 elements of the slice
  constexpr int kDpUnroll = 4;
  for (int64_t i0 = s0 + tid; i0 < s1; i0 += kDpUnroll * nth) {
    float4 gs[kDpUnroll];
#pragma unroll
    for (int u = 0; u < kDpUnroll; ++u) {
      const int64_t i = i0 + u * nth;
      gs[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i >= s1) continue;
      if (pr.grads_mc) {
        gs[u] = multimem_ld_reduce_add(pr.grads_mc + 4 * i);
      } else {
        for (int r = 0; r < world; ++r) {  // fixed order: every rank would get the same bits
          const float4 t = __ldcg(reinterpret_cast<const float4*>(pr.grads[r] + 4 * i));  // L2 (coherence point), not L1
          gs[u].x += t.x; gs[u].y += t.y; gs[u].z += t.z; gs[u].w += t.w;
        }
      }
    }
#pragma unroll
    for (int u = 0; u < kDpUnroll; ++u) {
      const int64_t i = i0 + u * nth;
      if (i >= s1) continue;
      const float4 g = gs[u];
      float4 pp = *reinterpret_cast<float4*>(pr.params[rank] + 4 * i);
      const int64_t j = i - s0;
      float4 mm = *reinterpret_cast<float4*>(m + 4 * j), vv = *reinterpret_cast<float4*>(v + 4 * j);
#define EIMS_ADAM1(P, G, Mm, V)                  \
  {                                              \
    float gr = G * k.grad_scale;                 \
    P *= k.decay;                                \
    Mm = Mm + (gr - Mm) * k.one_minus_b1;        \
    V = V * k.b2 + k.one_minus_b2 * gr * gr;     \
    float den = sqrtf(V) * k.inv_bc2_sqrt + k.eps; \
    P = P - k.step_size * (Mm / den);            \
  }
      EIMS_ADAM1(pp.x, g.x, mm.x, vv.x) EIMS_ADAM1(pp.y, g.y, mm.y, vv.y)
      EIMS_ADAM1(pp.z, g.z, mm.z, vv.z) EIMS_ADAM1(pp.w, g.w, mm.w, vv.w)
#undef EIMS_ADAM1
      *reinterpret_cast<float4*>(m + 4 * j) = mm;
      *reinterpret_cast<float4*>(v + 4 * j) = vv;
      if (pr.params_mc) {
        multimem_st(pr.params_mc + 4 * i, pp);
      } else {
        for (int r = 0; r < world; ++r) *reinterpret_cast<float4*>(pr.params[r] + 4 * i) = pp;
      }
    }
  }
  // the other gradient buffer (read by the peers during the previous step, which every rank has
  // left - they all passed phase 0 of this step) is zeroed for the step after this one
  if (zero_buf)
    for (int64_t i = base4 + tid; i < base4 + n4; i += nth)
      *reinterpret_cast<float4*>(zero_buf + 4 * i) = make_float4(0.f, 0.f, 0.f, 0.f);
  // ---- phase 2: when the whole grid has stored its slice, signal; the last block leaves only
  // after every rank's slice has landed in this rank's parameters
  __threadfence_system();
  if (!last_block_ticket(ticket, gridDim.x)) return;
  if ((int)threadIdx.x < world) st_release_sys(pr.signals[threadIdx.x] + (2 * row + 1) * kMaxRanks + rank, seq);
  wait_all(my_pad, 2 * row + 1, world, seq, timeout_ns, status);
}

}  // namespace eims

using namespace eims;

#pragma GCC visibility push(default)
extern "C" int eims_dp_adamw_fused(int32_t rank, int32_t world, const uint64_t* grad_ptrs, const uint64_t* param_ptrs,
                                   const uint64_t* signal_ptrs, uint64_t grads_multicast, uint64_t params_multicast,
                                   float* m_slice, float* v_slice, float* zero_buf, int64_t range_off,
                                   int64_t range_len, const eims_step* s, uint32_t seq, int32_t bucket,
                                   uint32_t* ticket, eims_stream_t stream) {
  return eims_dp_adamw_fused_blk(rank, world, grad_ptrs, param_ptrs, signal_ptrs, grads_multicast, params_multicast, m_slice,
                                 v_slice, zero_buf, range_off, range_len, s, seq, bucket, ticket, nullptr, stream);
}

extern "C" int eims_dp_adamw_fused_blk(int32_t rank, int32_t world, const uint64_t* grad_ptrs, const uint64_t* param_ptrs,
                                       const uint64_t* signal_ptrs, uint64_t grads_multicast, uint64_t params_multicast,
                                       float* m_slice, float* v_slice, float* zero_buf, int64_t range_off,
                                       int64_t range_len, const eims_step* s, uint32_t seq, int32_t bucket,
                                       uint32_t* ticket, const void* step_block, eims_stream_t stream) {
  if (world < 1 || world > kMaxRanks || rank < 0 || rank >= world || !grad_ptrs || !param_ptrs || !signal_ptrs ||
      (!step_block && (!s || s->step < 1)) || range_off < 0 || range_off % 4 || range_len <= 0 || range_len % (4 * (int64_t)world) || bucket < 0 ||
      bucket > 3 || !ticket)
    return EIMS_ERR_ARG;
  DpPeers pr{};
  for (int r = 0; r < world; ++r) {
    pr.grads[r] = reinterpret_cast<float*>(grad_ptrs[r]);
    pr.params[r] = reinterpret_cast<float*>(param_ptrs[r]);
    pr.signals[r] = reinterpret_cast<uint32_t*>(signal_ptrs[r]);
  }
  pr.grads_mc = reinterpret_cast<float*>(grads_multicast);
  pr.params_mc = reinterpret_cast<float*>(params_multicast);
  const AdamK k = step_block ? AdamK{} : make_adam_k(s);
  static unsigned long long timeout_ns = 0;
  if (!timeout_ns) {
    const char* e = getenv("EIMS_DP_TIMEOUT_S");
    const double sec = e ? atof(e) : 600.0;
    timeout_ns = (unsigned long long)((sec > 0.001 ? sec : 0.001) * 1e9);
  }
  const int64_t n4 = range_len / 4, per = n4 / world;
  int64_t blocks = (n4 + 255) / 256;   // the zeroing pass covers the whole range
  if (blocks > 148) blocks = 148;  // one block per SM
  // An early bucket (bucket > 0: exchanged on a side stream while the GraphConv layers are still being differentiated)
  // runs NEXT TO the backward kernels, and every one of its blocks spins in wait_all until the slowest peer arrives:
  // with a block on every SM it took more from the backward pass than the overlap gave back (0.3558 vs 0.3473 ms per
  // step at N=2).  A handful of blocks is plenty for ~0.5 MB per rank with ~130 us of backward to hide under.
  constexpr int kEarlyBlocks = 16;
  if (bucket > 0 && blocks > kEarlyBlocks) blocks = kEarlyBlocks;
  launch_pdl(dp_adamw_kernel, dim3((unsigned)blocks), dim3(256), 0, (cudaStream_t)stream, pr, rank, world, m_slice, v_slice,
             zero_buf, range_off / 4, n4, per, seq, (int)bucket, ticket, k, reinterpret_cast<const StepBlock*>(step_block),
             timeout_ns);
  return cudaPeekAtLastError() == cudaSuccess ? 0 : EIMS_ERR_CUDA;
}
#pragma GCC visibility pop

EIMS_TIMELINE_READER(dp_fused)
