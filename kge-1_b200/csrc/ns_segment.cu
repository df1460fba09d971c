// Negative-sampling backward without materialised candidate-gradient rows (SURVEY.md 8a a20 / 8d C3; tuning path of
// trainer.FusedNegSamplingStepper(segment_bwd=True); run by the GPU suite, tests/test_gpu_aux.py and
// tests/test_gpu_negative_sampling_exact.py).
//
// The default path (rows.cu pairs_bwd_kernel + update.cu sorted scatter) writes one gradient row per scored pair --
// dC [B*(1+N), d], 135 MB per slot at the WN18RR shape -- and the scatter reads it back.  But a candidate's gradient row
// is a function of (G[pair], Q[row(pair)], table[cand]) only, and Q (B rows) lives in L2.  So:
//   ns_bwd_q      dQ[row] = sum_j dscore/dq            (block per query row, as before, no dC)
//   ns_cand_grad  sort the pairs by candidate id (stable radix sort of (id, position)), run-length encode, then ONE WARP
//                 PER DISTINCT CANDIDATE walks its occurrences in position order, recomputes each occurrence's row from Q
//                 and the candidate's own row (read once) and adds the sum to the dense gradient: single writer per row,
//                 fixed order -> deterministic; traffic = the sorted index list + one table row per distinct candidate.
// Formulas per pair kind as in rows.cu (pairs_bwd_kernel): with g = dL/dscore,
//   DOT      dq += g c            dc  = g q
//   NEG_L1   dq -= g sgn(q - c)   dc  = g sgn(q - c)
//   NEG_L2   dq -= g (q-c)/dist   dc  = g (q-c)/dist      (dist = |score|; 0 -> 0)
//   ROT_L2   dq += g (q-c)/dist   dc  = -g (q-c)/dist
//   ROT_L1   per complex coordinate (k, k+h): m = |q-c|;  dq += g (q-c)/m, dc = -g (q-c)/m   (m = 0 -> 0)
#include <cstdint>

#include <cub/cub.cuh>

#include "common.cuh"

namespace kgeb {

constexpr int kNsWarps = 8;

// contribution of one pair to dq (sign as above) for coordinate k (ROT_L1: k < h handles (k, k+h))
template <int KIND>
__device__ __forceinline__ void pair_terms(float g, float coef, const float* __restrict__ q, const float* __restrict__ c,
                                           int k, int h, float& t0, float& t1) {
  t1 = 0.f;
  if (KIND == KGEB_DOT) {
    t0 = g * c[k];
  } else if (KIND == KGEB_NEG_L1) {
    t0 = -g * sgnf(q[k] - c[k]);
  } else if (KIND == KGEB_NEG_L2 || KIND == KGEB_ROT_L2) {
    t0 = coef * (q[k] - c[k]);
  } else {  // ROT_L1
    const float re = q[k] - c[k], im = q[k + h] - c[k + h];
    const float m = sqrtf(re * re + im * im);
    const float inv = m == 0.f ? 0.f : g / m;
    t0 = re * inv;
    t1 = im * inv;
  }
}

template <int KIND>
__global__ void __launch_bounds__(kNsWarps * 32)
ns_bwd_q_kernel(const float* __restrict__ Q, const float* __restrict__ table, const int64_t* __restrict__ cand, int64_t B,
                int64_t M, int d, const float* __restrict__ G, const float* __restrict__ scores, float* __restrict__ dQ) {
  extern __shared__ float smem[];  // [kNsWarps][d]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int h = d >> 1;
  const int kend = KIND == KGEB_ROT_L1 ? h : d;
  const int64_t row = blockIdx.x;
  const float* q = Q + row * d;
  float* acc = smem + warp * d;
  for (int k = lane; k < d; k += 32) acc[k] = 0.f;
  __syncwarp();
  for (int64_t j = warp; j < M; j += kNsWarps) {
    const int64_t pair = row * M + j;
    const float g = G[pair];
    const float* c = table + cand[pair] * (int64_t)d;
    float coef = 0.f;
    if (KIND == KGEB_NEG_L2 || KIND == KGEB_ROT_L2) {
      const float dist = fabsf(scores[pair]);
      coef = dist == 0.f ? 0.f : ((KIND == KGEB_NEG_L2 ? -g : g) / dist);
    }
    for (int k = lane; k < kend; k += 32) {
      float t0, t1;
      pair_terms<KIND>(g, coef, q, c, k, h, t0, t1);
      acc[k] += t0;
      if (KIND == KGEB_ROT_L1) acc[k + h] += t1;
    }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < d; k += blockDim.x) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < kNsWarps; ++w) s += smem[w * d + k];   // fixed order
    dQ[row * d + k] = s;
  }
}

// ids outside [0, vocab) are mapped to the sentinel key `vocab` (the sort covers vocab + 1 values): they form ONE run
// that the gradient kernel skips, instead of interleaving with the valid ids that share their low bits and splitting
// those runs (two warps adding to one dense row)
__global__ void ns_pack_kernel(const int64_t* __restrict__ cand, int64_t n, int64_t vocab, int32_t* __restrict__ keys,
                               int32_t* __restrict__ pos) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t e = cand[i];
  keys[i] = (e < 0 || e >= vocab) ? (int32_t)vocab : (int32_t)e;
  pos[i] = (int32_t)i;
}

// one warp per distinct candidate (run of the sorted id list); occurrences in ascending pair position
template <int KIND>
__global__ void __launch_bounds__(256)
ns_cand_grad_kernel(const float* __restrict__ Q, const float* __restrict__ table, int64_t M, int d,
                    const float* __restrict__ G, const float* __restrict__ scores, const int32_t* __restrict__ uniq,
                    const int32_t* __restrict__ run_off, const int32_t* __restrict__ num_runs, int64_t max_runs,
                    const int32_t* __restrict__ pos_sorted, int64_t vocab, float* __restrict__ dense) {
  const int lane = threadIdx.x & 31;
  const int64_t run = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (run >= max_runs || run >= *num_runs) return;
  const int64_t e = uniq[run];
  if (e < 0 || e >= vocab) return;
  const int h = d >> 1;
  const float* c = table + e * (int64_t)d;
  // registers: a0[i] = coordinate lane + 32 i (i < 4); a1[i] = its imaginary partner k + h (ROT_L1) or coordinate
  // lane + 32 (i + 4) of a wide row (the other kinds); d <= 256
  float a0[4] = {0.f, 0.f, 0.f, 0.f}, a1[4] = {0.f, 0.f, 0.f, 0.f};
  const int o0 = run_off[run], o1 = run_off[run + 1];
  for (int o = o0; o < o1; ++o) {
    const int64_t pair = pos_sorted[o];
    const float g = G[pair];
    const float* q = Q + (pair / M) * (int64_t)d;
    float coef = 0.f;
    if (KIND == KGEB_NEG_L2 || KIND == KGEB_ROT_L2) {
      const float dist = fabsf(scores[pair]);
      coef = dist == 0.f ? 0.f : ((KIND == KGEB_NEG_L2 ? -g : g) / dist);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int k = lane + 32 * i;
      float t0, t1;
      if (KIND == KGEB_ROT_L1) {
        if (k < h) {
          pair_terms<KIND>(g, coef, q, c, k, h, t0, t1);
          a0[i] -= t0;   // the candidate's gradient is the negative of the dq term
          a1[i] -= t1;
        }
      } else if (KIND == KGEB_DOT) {
        if (k < d) a0[i] += g * q[k];
        if (k + 128 < d) a1[i] += g * q[k + 128];
      } else {
        if (k < d) { pair_terms<KIND>(g, coef, q, c, k, h, t0, t1); a0[i] -= t0; }
        if (k + 128 < d) { pair_terms<KIND>(g, coef, q, c, k + 128, h, t0, t1); a1[i] -= t0; }
      }
    }
  }
  float* out = dense + e * (int64_t)d;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int k = lane + 32 * i;
    if (KIND == KGEB_ROT_L1) {
      if (k < h) {
        out[k] += a0[i];
        out[k + h] += a1[i];
      }
    } else {
      if (k < d) out[k] += a0[i];
      if (k + 128 < d) out[k + 128] += a1[i];
    }
  }
}

__global__ void ns_offsets_kernel(const int32_t* __restrict__ counts, const int32_t* __restrict__ num_runs, int32_t* off) {
  // exclusive scan of the run lengths by one block (runs <= n; serial per 1024-chunk with a running base)
  __shared__ int32_t base;
  if (threadIdx.x == 0) base = 0;
  __syncthreads();
  using Scan = cub::BlockScan<int32_t, 1024>;
  __shared__ typename Scan::TempStorage tmp;
  const int n = *num_runs;
  for (int start = 0; start < n; start += 1024) {
    const int i = start + threadIdx.x;
    const int32_t v = i < n ? counts[i] : 0;
    int32_t ex, total;
    Scan(tmp).ExclusiveSum(v, ex, total);
    if (i < n) off[i] = base + ex;
    __syncthreads();
    if (threadIdx.x == 0) base += total;
    __syncthreads();
  }
  if (threadIdx.x == 0) off[n] = base;
}

static inline size_t a256(size_t x) { return (x + 255) & ~(size_t)255; }

struct NsLayout {
  size_t keys_in, keys_out, pos_in, pos_out, uniq, counts, off, num_runs, cub, cub_bytes, total;
};
static NsLayout ns_layout(int64_t n) {
  NsLayout l;
  size_t sort_bytes = 0, rle_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const int32_t*)nullptr, (int32_t*)nullptr, (const int32_t*)nullptr,
                                  (int32_t*)nullptr, (int)n);
  cub::DeviceRunLengthEncode::Encode(nullptr, rle_bytes, (const int32_t*)nullptr, (int32_t*)nullptr, (int32_t*)nullptr,
                                     (int32_t*)nullptr, (int)n);
  size_t o = 0;
  l.keys_in = o; o += a256((size_t)n * 4);
  l.keys_out = o; o += a256((size_t)n * 4);
  l.pos_in = o; o += a256((size_t)n * 4);
  l.pos_out = o; o += a256((size_t)n * 4);
  l.uniq = o; o += a256((size_t)n * 4);
  l.counts = o; o += a256((size_t)n * 4);
  l.off = o; o += a256((size_t)(n + 1) * 4);
  l.num_runs = o; o += 256;
  l.cub = o;
  l.cub_bytes = sort_bytes > rle_bytes ? sort_bytes : rle_bytes;
  o += a256(l.cub_bytes);
  l.total = o;
  return l;
}

}  // namespace kgeb

using namespace kgeb;

#define NS_DISPATCH(kind, EXPR)                                          \
  switch (kind) {                                                        \
    case KGEB_DOT: { constexpr int K_ = KGEB_DOT; EXPR; } break;         \
    case KGEB_NEG_L1: { constexpr int K_ = KGEB_NEG_L1; EXPR; } break;   \
    case KGEB_NEG_L2: { constexpr int K_ = KGEB_NEG_L2; EXPR; } break;   \
    case KGEB_ROT_L1: { constexpr int K_ = KGEB_ROT_L1; EXPR; } break;   \
    default: { constexpr int K_ = KGEB_ROT_L2; EXPR; } break;            \
  }

extern "C" {

int kgeb_ns_bwd_q(int kind, const float* Q, const float* table, const int64_t* cand, int64_t B, int64_t M, int d,
                  const float* G, const float* scores, float* dQ, void* stream) {
  KGEB_REQUIRE(kind >= KGEB_DOT && kind <= KGEB_ROT_L2, "ns_bwd_q: unknown kind %d", kind);
  KGEB_REQUIRE(Q && table && cand && G && dQ && B >= 0 && M >= 0 && d > 0, "ns_bwd_q: bad arguments");
  KGEB_REQUIRE(!(kind == KGEB_NEG_L2 || kind == KGEB_ROT_L2) || scores, "ns_bwd_q: L2 kinds need the scores");
  KGEB_REQUIRE(!(kind >= KGEB_ROT_L1) || (d % 2 == 0), "RotatE requires embeddings of even dimensionality");
  if (B == 0) return KGEB_OK;
  const size_t smem = (size_t)kNsWarps * d * sizeof(float);
  KGEB_REQUIRE(smem <= 48 * 1024, "ns_bwd_q: dim %d too large", d);
  cudaStream_t st = as_stream(stream);
  NS_DISPATCH(kind, (ns_bwd_q_kernel<K_><<<(unsigned)B, kNsWarps * 32, smem, st>>>(Q, table, cand, B, M, d, G, scores, dQ)));
  KGEB_LAUNCH_CHECK("ns_bwd_q");
  return KGEB_OK;
}

int64_t kgeb_ns_segment_workspace_bytes(int64_t n) {
  if (n < 0 || n >= ((int64_t)1 << 31)) return -1;
  return (int64_t)ns_layout(n < 1 ? 1 : n).total;
}

int kgeb_ns_cand_grad(int kind, const float* Q, const float* table, const int64_t* cand, int64_t B, int64_t M, int d,
                      const float* G, const float* scores, int64_t vocab, float* dense, void* workspace,
                      int64_t workspace_bytes, void* stream) {
  KGEB_REQUIRE(kind >= KGEB_DOT && kind <= KGEB_ROT_L2, "ns_cand_grad: unknown kind %d", kind);
  KGEB_REQUIRE(Q && table && cand && G && dense && workspace && B >= 0 && M >= 0 && d > 0, "ns_cand_grad: bad arguments");
  KGEB_REQUIRE(d <= 256, "ns_cand_grad: dim %d too large (<= 256)", d);
  KGEB_REQUIRE(!(kind == KGEB_NEG_L2 || kind == KGEB_ROT_L2) || scores, "ns_cand_grad: L2 kinds need the scores");
  KGEB_REQUIRE(!(kind >= KGEB_ROT_L1) || (d % 2 == 0), "RotatE requires embeddings of even dimensionality");
  KGEB_REQUIRE(vocab > 0 && vocab < ((int64_t)1 << 31) - 1, "ns_cand_grad: vocabulary size out of range");
  const int64_t n = B * M;
  if (n == 0) return KGEB_OK;
  KGEB_REQUIRE(n < ((int64_t)1 << 31), "ns_cand_grad: too many pairs");
  const NsLayout l = ns_layout(n);
  KGEB_REQUIRE(workspace_bytes >= (int64_t)l.total, "ns_cand_grad: workspace too small");
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  int32_t* keys_in = reinterpret_cast<int32_t*>(ws + l.keys_in);
  int32_t* keys_out = reinterpret_cast<int32_t*>(ws + l.keys_out);
  int32_t* pos_in = reinterpret_cast<int32_t*>(ws + l.pos_in);
  int32_t* pos_out = reinterpret_cast<int32_t*>(ws + l.pos_out);
  int32_t* uniq = reinterpret_cast<int32_t*>(ws + l.uniq);
  int32_t* counts = reinterpret_cast<int32_t*>(ws + l.counts);
  int32_t* off = reinterpret_cast<int32_t*>(ws + l.off);
  int32_t* num_runs = reinterpret_cast<int32_t*>(ws + l.num_runs);
  cudaStream_t st = as_stream(stream);
  ns_pack_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(cand, n, vocab, keys_in, pos_in);
  KGEB_LAUNCH_CHECK("ns_pack");
  int bits = 1;
  while (bits < 31 && ((int64_t)1 << bits) < vocab + 1) ++bits;
  size_t cub_bytes = l.cub_bytes;
  cudaError_t e = cub::DeviceRadixSort::SortPairs(ws + l.cub, cub_bytes, keys_in, keys_out, pos_in, pos_out, (int)n, 0, bits, st);
  if (e != cudaSuccess) return cuda_status(e, "ns_cand_grad sort");
  cub_bytes = l.cub_bytes;
  e = cub::DeviceRunLengthEncode::Encode(ws + l.cub, cub_bytes, keys_out, uniq, counts, num_runs, (int)n, st);
  if (e != cudaSuccess) return cuda_status(e, "ns_cand_grad run-length encode");
  ns_offsets_kernel<<<1, 1024, 0, st>>>(counts, num_runs, off);
  KGEB_LAUNCH_CHECK("ns_offsets");
  NS_DISPATCH(kind, (ns_cand_grad_kernel<K_><<<(unsigned)((n + 7) / 8), 256, 0, st>>>(Q, table, M, d, G, scores, uniq, off,
                                                                                    num_runs, n, pos_out, vocab, dense)));
  KGEB_LAUNCH_CHECK("ns_cand_grad");
  return KGEB_OK;
}

}  // extern "C"
