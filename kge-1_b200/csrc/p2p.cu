// Data-parallel gradient exchange fused with the Adagrad update over NVLink peer memory (SURVEY.md 8e, "replicas" row).
//
// For graphs too small to shard (FB15k-237: a 7.4 MB table) every GPU of the box trains on its own batch against a
// full replica and the replicas exchange the dense gradient of both tables every step.  NCCL's all-reduce followed by
// a separate Adagrad kernel costs a collective launch, an all-reduce (reduce-scatter + all-gather of GRADIENTS) and a
// full-table update on every rank.  Here the exchange IS the update, one kernel per table over peer-mapped buffers
// (torch symmetric memory: cuMem VMM allocations mapped into every process of the node; NVSwitch gives every pair of
// GPUs full bandwidth):
//
//   barrier A            every rank's gradient buffer is complete
//   reduce+update        rank r owns the slice [lo_r, hi_r) of the table: it reads that slice of the gradient from all
//                        ranks (P2P loads, summed in rank order -> bit-identical on every replica), applies the Adagrad
//                        step to its slice of parameters and state (the state is therefore SHARDED: 1/world of it is
//                        touched per rank) and pushes the new parameter values into every peer's staging buffer (P2P
//                        stores): the all-gather moves updated WEIGHTS, the gradient never makes a second trip
//   barrier B            all pushes have landed
//   apply                each rank copies the other owners' slices from its staging buffer into its table (+ bf16
//                        mirror); the summed loss is read from the peers directly
//
// All four are plain kernels with peer pointers, so the whole step (compute + exchange) is ONE CUDA graph.  Per rank and
// step 2 * (world-1)/world * table bytes cross NVLink -- what a ring all-reduce moves -- with no second kernel pass over
// the gradient and a world-times smaller optimizer pass.
//
// Barriers: signal pad of rank k = uint32 slots [world]; at epoch e rank r stores e into slot r of every peer's pad
// (release, system scope) and spins until all its own slots reached e (acquire, system scope).  Epochs only grow, so a
// fast peer that already entered the next barrier (slot = e + 1) still satisfies ">= e"; no reset, no ABA.
#include <cstdint>

#include <cuda_bf16.h>

#include "common.cuh"

namespace kgeb {

constexpr int kMaxWorld = 16;

struct PeerPtrs {
  void* p[kMaxWorld];
};

__device__ __forceinline__ void st_release_sys(uint32_t* addr, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* addr) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(addr) : "memory");
  return v;
}

// Barrier inside a kernel: block 0 signals (this GPU has finished everything that precedes this kernel on its stream),
// every block waits until all peers signalled epoch e.  Bounded spin (~10 s): a dead peer must not hang the GPU.
__device__ __forceinline__ bool grid_peer_barrier(const PeerPtrs& pads, int rank, int world, uint32_t e, uint32_t* timeout_flag) {
  const int t = threadIdx.x;
  // sticky: once any barrier of this exchange has timed out, every later kernel returns before it writes anything
  // (weights, optimizer state, the step counter stay as they were; the host sees the flag with the next loss read-back)
  int bad = (*reinterpret_cast<volatile uint32_t*>(timeout_flag) != 0u);
  if (blockIdx.x == 0 && t < world && !bad) {
    __threadfence_system();
    st_release_sys(reinterpret_cast<uint32_t*>(pads.p[t]) + rank, e);
  }
  if (t < world && !bad) {
    const uint32_t* mine = reinterpret_cast<const uint32_t*>(pads.p[rank]) + t;
    long long spins = 0;
    while ((int32_t)(ld_acquire_sys(mine) - e) < 0) {
      __nanosleep(32);
      if (++spins > (1ll << 23)) {
        *reinterpret_cast<volatile uint32_t*>(timeout_flag) = 1u;
        bad = 1;
        break;
      }
    }
  }
  return __syncthreads_or(bad) == 0;
}

__host__ __device__ inline void slice_of(int64_t numel, int world, int r, int64_t& lo, int64_t& hi) {
  const int64_t per = ((numel + 4 * (int64_t)world - 1) / (4 * (int64_t)world)) * 4;   // multiple of 4 elements
  lo = per * r < numel ? per * r : numel;
  hi = lo + per < numel ? lo + per : numel;
}

struct Table {
  float* W;
  float* state;
  __nv_bfloat16* mirror;   // or NULL
  int64_t numel;           // multiple of 4
  int64_t flat_off;        // offset of this table's gradient in the exchanged flat buffer / of its weights in staging
};

__device__ __forceinline__ void adagrad4(float4& w, float4& s, const float4& g, float clr, float eps) {
  s.x = fmaf(g.x, g.x, s.x); s.y = fmaf(g.y, g.y, s.y); s.z = fmaf(g.z, g.z, s.z); s.w = fmaf(g.w, g.w, s.w);
  w.x -= clr * g.x / (sqrtf(s.x) + eps);
  w.y -= clr * g.y / (sqrtf(s.y) + eps);
  w.z -= clr * g.z / (sqrtf(s.z) + eps);
  w.w -= clr * g.w / (sqrtf(s.w) + eps);
}
__device__ __forceinline__ void store_bf16x4(__nv_bfloat16* dst, const float4& w) {
  __nv_bfloat162 a = __floats2bfloat162_rn(w.x, w.y), b = __floats2bfloat162_rn(w.z, w.w);
  uint2 o;
  o.x = *reinterpret_cast<uint32_t*>(&a);
  o.y = *reinterpret_cast<uint32_t*>(&b);
  *reinterpret_cast<uint2*>(dst) = o;
}

constexpr int kUnroll = 4;   // independent float4 groups per thread: remote loads are ~2 us away, keep many in flight

// Exchange kernel.  epoch counter *ctr = number of completed steps; this kernel's barrier uses 2*ctr + 1.
//   flat.p[k]  : rank k's [g_table0 | g_table1 | ... | loss] buffer;  stage.p[k] : rank k's [W_table0 | W_table1 ...]
__global__ void __launch_bounds__(256)
p2p_exchange_kernel(PeerPtrs pads, PeerPtrs flat, PeerPtrs stage, int rank, int world, const uint32_t* __restrict__ ctr,
                    uint32_t* timeout_flag, Table t0, Table t1, int64_t loss_off, float* __restrict__ loss_out, float clr_val,
                    float eps, const float* __restrict__ clr_dev) {
  if (!grid_peer_barrier(pads, rank, world, 2u * *ctr + 1u, timeout_flag)) return;   // every rank's gradients are complete
  if (blockIdx.x == 0 && threadIdx.x == 0 && loss_out) {
    float a = 0.f;
    for (int k = 0; k < world; ++k) a += reinterpret_cast<const float*>(flat.p[k])[loss_off];
    *loss_out = a;
  }
#pragma unroll 1
  for (int ti = 0; ti < 2; ++ti) {
    const Table& tb = ti == 0 ? t0 : t1;
    if (tb.numel == 0) continue;
    const float clr = clr_dev ? clr_dev[ti] : clr_val;   // _sched entry: one rate word per table
    int64_t lo, hi;
    slice_of(tb.numel, world, rank, lo, hi);
    const int64_t n4 = (hi - lo) / 4;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t q0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q0 < n4; q0 += stride * kUnroll) {
      float4 g[kUnroll];
#pragma unroll
      for (int u = 0; u < kUnroll; ++u) g[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int k = 0; k < world; ++k) {         // rank order: the same sum whichever rank owns the slice
        const float* src = reinterpret_cast<const float*>(flat.p[k]) + tb.flat_off + lo;
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
          const int64_t q = q0 + u * stride;
          if (q < n4) {
            const float4 h = *reinterpret_cast<const float4*>(src + q * 4);
            g[u].x += h.x; g[u].y += h.y; g[u].z += h.z; g[u].w += h.w;
          }
        }
      }
#pragma unroll
      for (int u = 0; u < kUnroll; ++u) {
        const int64_t q = q0 + u * stride;
        if (q >= n4) continue;
        const int64_t i = lo + q * 4;
        float4 w = *reinterpret_cast<float4*>(tb.W + i);
        float4 s = *reinterpret_cast<float4*>(tb.state + i);
        adagrad4(w, s, g[u], clr, eps);
        *reinterpret_cast<float4*>(tb.W + i) = w;
        *reinterpret_cast<float4*>(tb.state + i) = s;
        if (tb.mirror) store_bf16x4(tb.mirror + i, w);
        for (int k = 0; k < world; ++k)
          if (k != rank) *reinterpret_cast<float4*>(reinterpret_cast<float*>(stage.p[k]) + tb.flat_off + i) = w;
      }
    }
  }
}

// Apply kernel: barrier 2*ctr + 2 (all pushes have landed), then the other owners' slices from the local staging
// buffer into the tables (+ mirror); the last block to finish advances *ctr (every block has read it by then).
__global__ void __launch_bounds__(256)
p2p_apply_kernel(PeerPtrs pads, const float* __restrict__ stage, int rank, int world, uint32_t* ctr, uint32_t* ticket,
                 uint32_t* timeout_flag, Table t0, Table t1) {
  if (!grid_peer_barrier(pads, rank, world, 2u * *ctr + 2u, timeout_flag)) return;   // nothing applied, *ctr not advanced
#pragma unroll 1
  for (int ti = 0; ti < 2; ++ti) {
    const Table& tb = ti == 0 ? t0 : t1;
    if (tb.numel == 0) continue;
    int64_t lo, hi;
    slice_of(tb.numel, world, rank, lo, hi);
    const int64_t n4 = tb.numel / 4;
    for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < n4; q += (int64_t)gridDim.x * blockDim.x) {
      const int64_t i = q * 4;
      if (i >= lo && i < hi) continue;          // own slice: updated in place by the exchange kernel
      const float4 w = *reinterpret_cast<const float4*>(stage + tb.flat_off + i);
      *reinterpret_cast<float4*>(tb.W + i) = w;
      if (tb.mirror) store_bf16x4(tb.mirror + i, w);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(ticket, 1u) == gridDim.x - 1) {
      *ticket = 0;
      *ctr = *ctr + 1;
    }
  }
}

// One-shot all-reduce of a small buffer over peer memory (the O(batch * d) exchanges of the row-sharded training step:
// query-side rows, row statistics, dQ -- 1 MB each at the Wikidata5M bench shape).  Every rank has written its partial
// into ITS symmetric buffer; after the barrier each rank reads all partials (P2P loads) and reduces them in rank order,
// so all ranks hold bit-identical results.  A plain kernel: it sits in the same CUDA graph as the compute around it (NCCL
// calls between separately captured graphs cost ~10x the transfer time in launch gaps at this size).
//   mode 0: sum.   mode 1: each float4 is a row statistic (max m, sum l relative to m, sum x, label dot): the combined
//   row is (M = max_k m_k, sum_k l_k exp(m_k - M), sum_k x_k, sum_k d_k) -- log-sum-exp partials of entity shards.
// The barrier epoch is a device counter the last block advances; buffers may be reused by the NEXT BUT ONE collective
// (a rank enters collective c + 1 only after its own reads of collective c finished, and nobody passes the barrier of
// c + 1 before every rank entered it).
__global__ void __launch_bounds__(256)
p2p_allreduce_kernel(PeerPtrs pads, PeerPtrs bufs, int rank, int world, uint32_t* epoch, uint32_t* ticket,
                     uint32_t* timeout_flag, int64_t n4, int mode, float* __restrict__ out) {
  const bool ok = grid_peer_barrier(pads, rank, world, *epoch + 1u, timeout_flag);
  if (ok) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
      float4 acc;
      if (mode == 0) {
        acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int k = 0; k < world; ++k) {
          const float4 v = reinterpret_cast<const float4*>(bufs.p[k])[i];
          acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
      } else {
        float4 v[kMaxWorld];
        float m = -INFINITY;
        for (int k = 0; k < world; ++k) {
          v[k] = reinterpret_cast<const float4*>(bufs.p[k])[i];
          m = fmaxf(m, v[k].x);
        }
        acc = make_float4(m, 0.f, 0.f, 0.f);
        for (int k = 0; k < world; ++k) {
          acc.y += v[k].x == -INFINITY ? 0.f : v[k].y * __expf(v[k].x - m);
          acc.z += v[k].z;
          acc.w += v[k].w;
        }
      }
      reinterpret_cast<float4*>(out)[i] = acc;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(ticket, 1u) == gridDim.x - 1) {
      *ticket = 0;
      if (ok) *epoch = *epoch + 1;
    }
  }
}

static int fill_ptrs(PeerPtrs& pp, const void* const* host_ptrs, int world) {
  for (int k = 0; k < kMaxWorld; ++k) pp.p[k] = k < world ? const_cast<void*>(host_ptrs[k]) : nullptr;
  return 0;
}

}  // namespace kgeb

using namespace kgeb;

extern "C" {

}  // extern "C"

// kgeb_p2p_exchange and its _sched sibling: one kernel, clr_dev == NULL selects the by-value rate of both tables
static int p2p_exchange(const void* const* peer_pads, const void* const* peer_flat, const void* const* peer_stage, int rank,
                        int world, const uint32_t* ctr, uint32_t* timeout_flag, float* W0, float* state0, void* mirror0,
                        int64_t numel0, float* W1, float* state1, int64_t numel1, float* loss_out, float clr,
                        const float* clr_dev, float eps, void* stream) {
  KGEB_REQUIRE(peer_pads && peer_flat && peer_stage && ctr && timeout_flag && W0 && state0 && numel0 >= 0 && numel1 >= 0 &&
                   (numel1 == 0 || (W1 && state1)) && world >= 1 && world <= kMaxWorld && rank >= 0 && rank < world,
               "p2p_exchange: bad arguments");
  KGEB_REQUIRE(numel0 % 4 == 0 && numel1 % 4 == 0, "p2p_exchange: table sizes must be multiples of 4 elements");
  PeerPtrs pads, flat, stage;
  fill_ptrs(pads, peer_pads, world);
  fill_ptrs(flat, peer_flat, world);
  fill_ptrs(stage, peer_stage, world);
  uintptr_t bits = reinterpret_cast<uintptr_t>(W0) | reinterpret_cast<uintptr_t>(state0) | reinterpret_cast<uintptr_t>(mirror0) |
                   reinterpret_cast<uintptr_t>(W1) | reinterpret_cast<uintptr_t>(state1);
  for (int k = 0; k < world; ++k) bits |= reinterpret_cast<uintptr_t>(flat.p[k]) | reinterpret_cast<uintptr_t>(stage.p[k]);
  KGEB_REQUIRE((bits & 15) == 0, "p2p_exchange: pointers must be 16-byte aligned");
  Table t0{W0, state0, reinterpret_cast<__nv_bfloat16*>(mirror0), numel0, 0};
  Table t1{W1, state1, nullptr, numel1, numel0};
  int64_t lo, hi;
  slice_of(numel0, world, rank, lo, hi);
  int64_t blocks = ((hi - lo) / 4 + 256 * kUnroll - 1) / (256 * kUnroll) + 1;
  const int grid = (int)(blocks > (int64_t)kNumSMs * 4 ? (int64_t)kNumSMs * 4 : blocks);   // all blocks co-resident
  p2p_exchange_kernel<<<grid, 256, 0, as_stream(stream)>>>(pads, flat, stage, rank, world, ctr, timeout_flag, t0, t1,
                                                          numel0 + numel1, loss_out, clr, eps, clr_dev);
  KGEB_LAUNCH_CHECK("p2p_exchange");
  return KGEB_OK;
}

extern "C" {

int kgeb_p2p_exchange(const void* const* peer_pads, const void* const* peer_flat, const void* const* peer_stage, int rank,
                      int world, const uint32_t* ctr, uint32_t* timeout_flag, float* W0, float* state0, void* mirror0,
                      int64_t numel0, float* W1, float* state1, int64_t numel1, float* loss_out, float clr, float eps,
                      void* stream) {
  return p2p_exchange(peer_pads, peer_flat, peer_stage, rank, world, ctr, timeout_flag, W0, state0, mirror0, numel0, W1,
                      state1, numel1, loss_out, clr, nullptr, eps, stream);
}

int kgeb_p2p_exchange_sched(const void* const* peer_pads, const void* const* peer_flat, const void* const* peer_stage,
                            int rank, int world, const uint32_t* ctr, uint32_t* timeout_flag, float* W0, float* state0,
                            void* mirror0, int64_t numel0, float* W1, float* state1, int64_t numel1, float* loss_out,
                            const float* clr, float eps, void* stream) {
  KGEB_REQUIRE(clr, "p2p_exchange_sched: the learning-rate words are NULL");
  return p2p_exchange(peer_pads, peer_flat, peer_stage, rank, world, ctr, timeout_flag, W0, state0, mirror0, numel0, W1,
                      state1, numel1, loss_out, 0.f, clr, eps, stream);
}

int kgeb_p2p_allreduce(const void* const* peer_pads, const void* const* peer_bufs, int rank, int world, uint32_t* epoch,
                       uint32_t* timeout_flag, int64_t numel, int mode, float* out, void* stream) {
  KGEB_REQUIRE(peer_pads && peer_bufs && epoch && timeout_flag && out && numel >= 0 && world >= 1 && world <= kMaxWorld &&
                   rank >= 0 && rank < world && (mode == 0 || mode == 1),
               "p2p_allreduce: bad arguments");
  KGEB_REQUIRE(numel % 4 == 0, "p2p_allreduce: the element count must be a multiple of 4");
  PeerPtrs pads, bufs;
  fill_ptrs(pads, peer_pads, world);
  fill_ptrs(bufs, peer_bufs, world);
  uintptr_t bits = reinterpret_cast<uintptr_t>(out);
  for (int k = 0; k < world; ++k) bits |= reinterpret_cast<uintptr_t>(bufs.p[k]);
  KGEB_REQUIRE((bits & 15) == 0, "p2p_allreduce: pointers must be 16-byte aligned");
  const int64_t n4 = numel / 4;
  int64_t blocks = (n4 + 255) / 256;
  if (blocks < 1) blocks = 1;
  const int grid = (int)(blocks > (int64_t)kNumSMs * 2 ? (int64_t)kNumSMs * 2 : blocks);
  p2p_allreduce_kernel<<<grid, 256, 0, as_stream(stream)>>>(pads, bufs, rank, world, epoch, epoch + 1, timeout_flag, n4,
                                                            mode, out);
  KGEB_LAUNCH_CHECK("p2p_allreduce");
  return KGEB_OK;
}

int kgeb_p2p_apply(const void* const* peer_pads, const float* stage, int rank, int world, uint32_t* ctr, uint32_t* ticket,
                   uint32_t* timeout_flag, float* W0, void* mirror0, int64_t numel0, float* W1, int64_t numel1,
                   void* stream) {
  KGEB_REQUIRE(peer_pads && stage && ctr && ticket && timeout_flag && W0 && numel0 >= 0 && numel1 >= 0 &&
                   (numel1 == 0 || W1) && world >= 1 && world <= kMaxWorld && rank >= 0 && rank < world,
               "p2p_apply: bad arguments");
  KGEB_REQUIRE(numel0 % 4 == 0 && numel1 % 4 == 0, "p2p_apply: table sizes must be multiples of 4 elements");
  PeerPtrs pads;
  fill_ptrs(pads, peer_pads, world);
  Table t0{W0, nullptr, reinterpret_cast<__nv_bfloat16*>(mirror0), numel0, 0};
  Table t1{W1, nullptr, nullptr, numel1, numel0};
  int64_t blocks = (numel0 / 4 + 255) / 256 + 1;
  const int grid = (int)(blocks > (int64_t)kNumSMs * 4 ? (int64_t)kNumSMs * 4 : blocks);
  p2p_apply_kernel<<<grid, 256, 0, as_stream(stream)>>>(pads, stage, rank, world, ctr, ticket, timeout_flag, t0, t1);
  KGEB_LAUNCH_CHECK("p2p_apply");
  return KGEB_OK;
}

}  // extern "C"
