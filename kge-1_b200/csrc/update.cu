// Embedding gradient scatter and optimizer row updates.
//  * sort-based, deterministic segment scatter-add (autograd of nn.Embedding in the reference,
//    embedder/lookup_embedder.py:39-41,91-92): CUB radix sort of (row id, position) -- a stable sort, so
//    equal ids keep ascending position order -- then one warp per distinct id sums its rows in that
//    fixed order.  No float atomics anywhere.
//  * Adagrad / Adam steps with torch.optim semantics (util/optimizer.py:10-17), dense and touched-rows.
//  * device-side key lookup over KvsAllIndex arrays (indexing.py:36-55).
#include "common.cuh"
#include <cub/cub.cuh>
#include <cuda_bf16.h>

namespace kgeb {

struct ScatterWs {
  float* part;  // [ceil(n/CHUNK)][2][d] partial segment sums
  int64_t* keys_in;
  int64_t* keys_out;
  int32_t* pos_in;
  int32_t* pos_out;
  int32_t* seg_id;     // inclusive scan of head flags (1-based segment number per sorted position)
  int32_t* seg_start;  // [n+1]
  void* cub_tmp;
  size_t cub_bytes;
};

static size_t align256(size_t x) { return (x + 255) / 256 * 256; }

static size_t cub_temp_bytes(int64_t n) {
  size_t a = 0, b = 0, c = 0, c2 = 0;
  cub::DeviceRadixSort::SortKeys(nullptr, c, (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)n);
  cub::DeviceRadixSort::SortKeys(nullptr, c2, (const uint64_t*)nullptr, (uint64_t*)nullptr, (int)n);
  if (c2 > c) c = c2;
  cub::DeviceRadixSort::SortPairs(nullptr, a, (const int64_t*)nullptr, (int64_t*)nullptr, (const int32_t*)nullptr,
                                  (int32_t*)nullptr, (int)n);
  cub::DeviceScan::InclusiveSum(nullptr, b, (const int32_t*)nullptr, (int32_t*)nullptr, (int)n);
  a = a > b ? a : b;
  return a > c ? a : c;
}

static size_t part_bytes(int64_t n, int d) { return align256((size_t)((n + 7) / 8) * 2 * (size_t)d * 4); }

static int64_t scatter_ws_bytes(int64_t n, int d) {
  if (n < 1) n = 1;
  return (int64_t)(2 * align256(n * 8) + 3 * align256((n + 1) * 4) + align256(cub_temp_bytes(n)) + part_bytes(n, d) + 512);
}

static bool carve(void* ws, int64_t bytes, int64_t n, int d, ScatterWs& w) {
  if (!ws || bytes < scatter_ws_bytes(n, d)) return false;
  char* p = reinterpret_cast<char*>(ws);
  p = reinterpret_cast<char*>(align256(reinterpret_cast<size_t>(p)));
  w.part = reinterpret_cast<float*>(p); p += part_bytes(n, d);
  w.keys_in = reinterpret_cast<int64_t*>(p); p += align256(n * 8);
  w.keys_out = reinterpret_cast<int64_t*>(p); p += align256(n * 8);
  w.pos_in = reinterpret_cast<int32_t*>(p); p += align256((n + 1) * 4);
  w.pos_out = reinterpret_cast<int32_t*>(p); p += align256((n + 1) * 4);
  w.seg_id = reinterpret_cast<int32_t*>(p); p += align256((n + 1) * 4);
  w.cub_tmp = p;
  w.cub_bytes = cub_temp_bytes(n);
  w.seg_start = w.pos_in;  // pos_in is dead after the sort; reuse it for the segment starts
  return true;
}

__global__ void iota_keys_kernel(const void* idx, int idx64, int64_t n, int64_t* keys, int32_t* pos) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) {
    keys[i] = load_index(idx, idx64, i);
    pos[i] = (int32_t)i;
  }
}
__global__ void head_flags_kernel(const int64_t* __restrict__ keys, int64_t n, int32_t* __restrict__ flags) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) flags[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1 : 0;
}
__global__ void seg_starts_kernel(const int64_t* __restrict__ keys, const int32_t* __restrict__ seg_id, int64_t n,
                                  int32_t* __restrict__ seg_start, int64_t* __restrict__ num_uniq) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) {
    if (i == 0 || keys[i] != keys[i - 1]) seg_start[seg_id[i] - 1] = (int32_t)i;
    if (i == n - 1) {
      seg_start[seg_id[i]] = (int32_t)n;
      if (num_uniq) *num_uniq = seg_id[i];
    }
  }
}

// Segment sums in two fixed-order phases (deterministic: every output element has exactly one writer per phase and
// a fixed summation order; hot keys are not walked serially):
//  phase 1: one warp per chunk of CHUNK consecutive sorted positions loads its rows in one batch and adds them in
//           position order; runs that are whole segments go straight to the output, the (at most two) runs that
//           continue into a neighbouring chunk go to part[chunk][0] (run continuing from the previous chunk) /
//           part[chunk][1] (run continuing into the next);
//  phase 2: one warp per segment that spans several chunks adds its partials in chunk order.
constexpr int CHUNK = 8;

__device__ __forceinline__ void seg_store(float4 acc, int c0, int d, float* dst, bool vec) {
  if (vec && c0 + 3 < d) {
    *reinterpret_cast<float4*>(dst) = acc;
  } else {
    float v[4] = {acc.x, acc.y, acc.z, acc.w};
    for (int j = 0; j < 4 && c0 + j < d; ++j) dst[j] = v[j];
  }
}
// dense[...] += acc.  Each address has a single writer in a kernel, so the fire-and-forget reduction is deterministic.
__device__ __forceinline__ void seg_add(float4 acc, int c0, int d, float* dst) {
  float v[4] = {acc.x, acc.y, acc.z, acc.w};
#pragma unroll
  for (int j = 0; j < 4; ++j)
    if (c0 + j < d) atomicAdd(dst + j, v[j]);
}

template <bool DENSE>
__global__ void __launch_bounds__(256)
segment_sum_phase1(const int64_t* __restrict__ keys, const int32_t* __restrict__ pos,
                   const int32_t* __restrict__ seg_id, int64_t n, int d, const float* __restrict__ rows,
                   float* __restrict__ dense, int64_t vocab, int64_t* __restrict__ uniq_ids,
                   float* __restrict__ uniq_rows, float* __restrict__ part) {
  const int lane = threadIdx.x & 31;
  const int64_t nchunks = (n + CHUNK - 1) / CHUNK;
  const bool vec = (d & 3) == 0;
  for (int64_t ch = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); ch < nchunks;
       ch += (int64_t)gridDim.x * (blockDim.x >> 5)) {
    const int64_t cb = ch * CHUNK;
    const int m = (int)min((int64_t)CHUNK, n - cb);
    // chunk metadata, one position per lane (all loads issued together)
    int my_pos = 0, my_sid = -1;
    int64_t my_key = 0;
    if (lane < m) {
      my_pos = pos[cb + lane];
      my_sid = seg_id[cb + lane];
      my_key = keys[cb + lane];
    }
    const int prev_sid = cb > 0 ? seg_id[cb - 1] : -1;
    const int next_sid = cb + m < n ? seg_id[cb + m] : -2;
    int sid[CHUNK], prw[CHUNK];
    int64_t key[CHUNK];
#pragma unroll
    for (int j = 0; j < CHUNK; ++j) {
      sid[j] = __shfl_sync(0xffffffffu, my_sid, j);
      prw[j] = __shfl_sync(0xffffffffu, my_pos, j);
      key[j] = __shfl_sync(0xffffffffu, my_key, j);
    }
    for (int cg = 0; cg < d; cg += 128) {
      const int c0 = cg + lane * 4;
      if (c0 >= d) continue;
      float4 v[CHUNK];
#pragma unroll
      for (int j = 0; j < CHUNK; ++j) {  // the whole chunk in flight at once
        v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (j < m) {
          const float* src = rows + (int64_t)prw[j] * d + c0;
          if (vec) {
            v[j] = __ldg(reinterpret_cast<const float4*>(src));
          } else {
            v[j].x = src[0];
            if (c0 + 1 < d) v[j].y = src[1];
            if (c0 + 2 < d) v[j].z = src[2];
            if (c0 + 3 < d) v[j].w = src[3];
          }
        }
      }
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      bool from_prev = (prev_sid == sid[0]);   // the current run continues a segment of the previous chunk
#pragma unroll
      for (int j = 0; j < CHUNK; ++j) {
        if (j < m) {
          acc.x += v[j].x; acc.y += v[j].y; acc.z += v[j].z; acc.w += v[j].w;
          const bool last_of_chunk = (j == m - 1);
          const bool run_ends = last_of_chunk || (sid[j + 1 < CHUNK ? j + 1 : j] != sid[j]);
          if (run_ends) {
            const bool to_next = last_of_chunk && (next_sid == sid[j]);
            if (!from_prev && !to_next) {          // a whole segment
              const int64_t k = key[j];
              if (DENSE) {
                if (k >= 0 && k < vocab) seg_add(acc, c0, d, dense + k * d + c0);
              } else {
                seg_store(acc, c0, d, uniq_rows + (int64_t)(sid[j] - 1) * d + c0, vec);
                if (cg == 0 && lane == 0) uniq_ids[sid[j] - 1] = k;
              }
            } else {
              seg_store(acc, c0, d, part + ((ch * 2 + (from_prev ? 0 : 1)) * (int64_t)d) + c0, vec);
            }
            acc = make_float4(0.f, 0.f, 0.f, 0.f);
            from_prev = false;
          }
        }
      }
    }
  }
}

template <bool DENSE>
__global__ void __launch_bounds__(256)
segment_sum_phase2(const int64_t* __restrict__ keys, const int32_t* __restrict__ seg_id,
                   const int32_t* __restrict__ seg_start, int64_t n, int d, float* __restrict__ dense, int64_t vocab,
                   int64_t* __restrict__ uniq_ids, float* __restrict__ uniq_rows, const float* __restrict__ part) {
  const int lane = threadIdx.x & 31;
  const int nseg = seg_id[n - 1];
  const bool vec = (d & 3) == 0;
  for (int64_t seg = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); seg < nseg;
       seg += (int64_t)gridDim.x * (blockDim.x >> 5)) {
    const int sb = seg_start[seg], se = seg_start[seg + 1];
    const int64_t c0ch = sb / CHUNK, c1ch = (se - 1) / CHUNK;
    if (c0ch == c1ch) continue;  // finished in phase 1
    const int64_t key = keys[sb];
    if (DENSE && (key < 0 || key >= vocab)) continue;
    for (int cg = 0; cg < d; cg += 128) {
      const int c0 = cg + lane * 4;
      if (c0 >= d) continue;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int64_t ch = c0ch; ch <= c1ch; ch += 8) {
        float4 v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {  // eight partials in flight, added in chunk order
          v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (ch + j <= c1ch) {
            const float* src = part + (((ch + j) * 2 + ((ch + j) == c0ch ? 1 : 0)) * (int64_t)d) + c0;
            if (vec && c0 + 3 < d) {
              v[j] = *reinterpret_cast<const float4*>(src);
            } else {
              v[j].x = src[0];
              if (c0 + 1 < d) v[j].y = src[1];
              if (c0 + 2 < d) v[j].z = src[2];
              if (c0 + 3 < d) v[j].w = src[3];
            }
          }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) { acc.x += v[j].x; acc.y += v[j].y; acc.z += v[j].z; acc.w += v[j].w; }
      }
      if (DENSE) seg_add(acc, c0, d, dense + key * d + c0);
      else seg_store(acc, c0, d, uniq_rows + seg * (int64_t)d + c0, vec);
    }
    if (!DENSE && lane == 0) uniq_ids[seg] = key;
  }
}

// ------------------------------------------------------------------------------------------
// small-n fast path of the dense scatter (n <= 32768 rows, the per-batch case): ids and positions packed into one
// 32-bit word (id << PB | position), ONE single-block radix sort over the id bits only (stable, so positions stay
// ascending within an id), then the two fixed-order phases working on the packed words -- 3 kernels instead of 11.
// ------------------------------------------------------------------------------------------
template <int ITEMS>
__global__ void __launch_bounds__(1024)
block_pack_sort_kernel(const void* idx, int idx64, int n, int pb, int kb, int presorted, uint32_t* __restrict__ packed) {
  using Sort = cub::BlockRadixSort<uint32_t, 1024, ITEMS>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  typename Sort::TempStorage& tmp = *reinterpret_cast<typename Sort::TempStorage*>(smem_raw);
  uint32_t keys[ITEMS];
#pragma unroll
  for (int j = 0; j < ITEMS; ++j) {
    const int i = threadIdx.x * ITEMS + j;  // blocked arrangement: ascending positions
    keys[j] = 0xFFFFFFFFu;                  // padding sorts last
    if (i < n) keys[j] = ((uint32_t)load_index(idx, idx64, i) << pb) | (uint32_t)i;
  }
  if (!presorted) Sort(tmp).Sort(keys, pb, pb + kb);
#pragma unroll
  for (int j = 0; j < ITEMS; ++j) {
    const int i = threadIdx.x * ITEMS + j;
    if (i < n) packed[i] = keys[j];
  }
}

template <typename W>
__global__ void __launch_bounds__(256)
packed_sum_phase1(const W* __restrict__ packed, int n, int pb, int d, const float* __restrict__ rows,
                  float* __restrict__ dense, int64_t vocab, float* __restrict__ part) {
  const int lane = threadIdx.x & 31;
  const int nchunks = (n + CHUNK - 1) / CHUNK;
  const bool vec = (d & 3) == 0;
  const W pmask = ((W)1 << pb) - (W)1;
  for (int ch = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); ch < nchunks; ch += gridDim.x * (blockDim.x >> 5)) {
    const int cb = ch * CHUNK;
    const int m = min(CHUNK, n - cb);
    W mine = ~(W)0;
    if (lane < m) mine = packed[cb + lane];
    const int64_t prev_key = cb > 0 ? (int64_t)(packed[cb - 1] >> pb) : -1;
    const int64_t next_key = cb + m < n ? (int64_t)(packed[cb + m] >> pb) : -2;
    int64_t key[CHUNK];
    int prw[CHUNK];
#pragma unroll
    for (int j = 0; j < CHUNK; ++j) {
      const W w = __shfl_sync(0xffffffffu, mine, j);
      key[j] = (int64_t)(w >> pb);
      prw[j] = (int)(w & pmask);
    }
    for (int cg = 0; cg < d; cg += 128) {
      const int c0 = cg + lane * 4;
      if (c0 >= d) continue;
      float4 v[CHUNK];
#pragma unroll
      for (int j = 0; j < CHUNK; ++j) {
        v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (j < m) {
          const float* src = rows + (int64_t)prw[j] * d + c0;
          if (vec) {
            v[j] = __ldg(reinterpret_cast<const float4*>(src));
          } else {
            v[j].x = src[0];
            if (c0 + 1 < d) v[j].y = src[1];
            if (c0 + 2 < d) v[j].z = src[2];
            if (c0 + 3 < d) v[j].w = src[3];
          }
        }
      }
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      bool from_prev = (prev_key == key[0]);
#pragma unroll
      for (int j = 0; j < CHUNK; ++j) {
        if (j < m) {
          acc.x += v[j].x; acc.y += v[j].y; acc.z += v[j].z; acc.w += v[j].w;
          const bool last_of_chunk = (j == m - 1);
          const bool run_ends = last_of_chunk || (key[j + 1 < CHUNK ? j + 1 : j] != key[j]);
          if (run_ends) {
            const bool to_next = last_of_chunk && (next_key == key[j]);
            if (!from_prev && !to_next) {
              if (key[j] >= 0 && key[j] < vocab) seg_add(acc, c0, d, dense + key[j] * d + c0);
            } else {
              seg_store(acc, c0, d, part + (((int64_t)ch * 2 + (from_prev ? 0 : 1)) * d) + c0, vec);
            }
            acc = make_float4(0.f, 0.f, 0.f, 0.f);
            from_prev = false;
          }
        }
      }
    }
  }
}

// one warp per chunk whose last run STARTS a segment that continues into the following chunks: it finds the end of
// the segment by binary search on the sorted ids and adds the partials in chunk order
template <typename W>
__global__ void __launch_bounds__(256)
packed_sum_phase2(const W* __restrict__ packed, int n, int pb, int d, float* __restrict__ dense, int64_t vocab,
                  const float* __restrict__ part) {
  const int lane = threadIdx.x & 31;
  const int nchunks = (n + CHUNK - 1) / CHUNK;
  const bool vec = (d & 3) == 0;
  for (int ch = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); ch < nchunks; ch += gridDim.x * (blockDim.x >> 5)) {
    const int cb = ch * CHUNK;
    const int m = min(CHUNK, n - cb);
    if (cb + m >= n) continue;                                  // nothing follows the last chunk
    const W kq = packed[cb + m - 1] >> pb;                      // id of the chunk's last run
    if ((packed[cb + m] >> pb) != kq) continue;                 // it does not continue
    if ((packed[cb] >> pb) == kq && cb > 0 && (packed[cb - 1] >> pb) == kq) continue;  // not the segment's first chunk
    // first position with id > kq: 32-ary search, one probe per lane and round
    int lo = cb + m, hi = n;
    while (hi - lo > 0) {
      const int span = hi - lo;
      const int step = (span + 31) / 32;
      const int probe = min(lo + (lane + 1) * step - 1, hi - 1);   // last position of this lane's slice
      const bool gt = (packed[probe] >> pb) > kq;
      const unsigned mask = __ballot_sync(0xffffffffu, gt);
      if (mask == 0) { lo = hi; break; }
      const int first = __ffs(mask) - 1;                           // slice containing the boundary
      const int nlo = lo + first * step;
      hi = min(lo + (first + 1) * step - 1, hi - 1);                // its last position has id > kq
      lo = nlo;
      if (step == 1) { lo = hi; break; }
    }
    const int c1 = (lo - 1) / CHUNK;
    if ((int64_t)kq >= vocab) continue;
    for (int cg = 0; cg < d; cg += 128) {
      const int c0 = cg + lane * 4;
      if (c0 >= d) continue;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int c = ch; c <= c1; c += 8) {
        float4 v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (c + j <= c1) {
            const float* src = part + (((int64_t)(c + j) * 2 + ((c + j) == ch ? 1 : 0)) * d) + c0;
            if (vec && c0 + 3 < d) {
              v[j] = *reinterpret_cast<const float4*>(src);
            } else {
              v[j].x = src[0];
              if (c0 + 1 < d) v[j].y = src[1];
              if (c0 + 2 < d) v[j].z = src[2];
              if (c0 + 3 < d) v[j].w = src[3];
            }
          }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) { acc.x += v[j].x; acc.y += v[j].y; acc.z += v[j].z; acc.w += v[j].w; }
      }
      seg_add(acc, c0, d, dense + (int64_t)kq * d + c0);
    }
  }
}

static int bits_for(int64_t x) {  // smallest b with 2^b >= x
  int b = 1;
  while (b < 62 && ((int64_t)1 << b) < x) ++b;
  return b;
}

template <typename W>
__global__ void pack_keys_kernel(const void* idx, int idx64, int n, int pb, W* __restrict__ packed) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) packed[i] = ((W)load_index(idx, idx64, i) << pb) | (W)i;
}

// packed words straight from a precomputed stable argsort of the ids (no device sort)
template <typename W>
__global__ void pack_perm_kernel(const void* idx, int idx64, const int32_t* __restrict__ perm, int n, int pb,
                                 W* __restrict__ packed) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    const int src = perm[i];
    packed[i] = ((W)load_index(idx, idx64, src) << pb) | (W)src;
  }
}

template <typename W>
static int packed_phases(const W* packed, int64_t n, int pb, int d, const float* rows, float* dense, int64_t vocab,
                         float* part, cudaStream_t st) {
  const int nchunks = (int)((n + CHUNK - 1) / CHUNK);
  int blocks = (nchunks + 7) / 8;
  if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
  packed_sum_phase1<W><<<blocks, 256, 0, st>>>(packed, (int)n, pb, d, rows, dense, vocab, part);
  packed_sum_phase2<W><<<blocks, 256, 0, st>>>(packed, (int)n, pb, d, dense, vocab, part);
  KGEB_LAUNCH_CHECK("packed scatter");
  return KGEB_OK;
}

// returns -1 when the packed path does not apply
static int scatter_small(const void* idx, int idx64, const float* rows, int64_t n, int d, float* dense, int64_t vocab,
                         ScatterWs& w, cudaStream_t st, bool presorted) {
  const int pb = bits_for(n), kb = bits_for(vocab);
  if (n > (1 << 26) || pb + kb > 62) return -1;
  if (pb + kb > 32) {
    // 64-bit words: coalesced pack, keys-only device radix sort over the id bits (stable -> positions ascending)
    uint64_t* packed = reinterpret_cast<uint64_t*>(w.keys_in);
    uint64_t* tmp = reinterpret_cast<uint64_t*>(w.keys_out);
    pack_keys_kernel<uint64_t><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(idx, idx64, (int)n, pb, presorted ? packed : tmp);
    if (!presorted) {
      size_t bytes = w.cub_bytes;
      cudaError_t e = cub::DeviceRadixSort::SortKeys(w.cub_tmp, bytes, tmp, packed, (int)n, pb, pb + kb, st);
      if (e != cudaSuccess) return cuda_status(e, "radix sort (packed64)");
    }
    return packed_phases<uint64_t>(packed, n, pb, d, rows, dense, vocab, w.part, st);
  }
  uint32_t* packed = reinterpret_cast<uint32_t*>(w.keys_in);
  if (n <= 8192) {
    using Sort = cub::BlockRadixSort<uint32_t, 1024, 8>;
    const int smem = (int)sizeof(typename Sort::TempStorage);
    cudaError_t e = cudaFuncSetAttribute(block_pack_sort_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return cuda_status(e, "block sort smem attribute");
    block_pack_sort_kernel<8><<<1, 1024, smem, st>>>(idx, idx64, (int)n, pb, kb, presorted, packed);
  } else {
    // multi-block: coalesced pack, then a keys-only device radix sort over the id bits (stable -> positions ascending)
    uint32_t* tmp = reinterpret_cast<uint32_t*>(w.keys_out);
    pack_keys_kernel<uint32_t><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(idx, idx64, (int)n, pb, presorted ? packed : tmp);
    if (!presorted) {
      size_t bytes = w.cub_bytes;
      cudaError_t e = cub::DeviceRadixSort::SortKeys(w.cub_tmp, bytes, tmp, packed, (int)n, pb, pb + kb, st);
      if (e != cudaSuccess) return cuda_status(e, "radix sort (packed)");
    }
  }
  return packed_phases<uint32_t>(packed, n, pb, d, rows, dense, vocab, w.part, st);
}

template <bool DENSE>
static int segment_sums(ScatterWs& w, int64_t n, int d, const float* rows, float* dense, int64_t vocab,
                        int64_t* uniq_ids, float* uniq_rows, cudaStream_t st) {
  const int64_t nchunks = (n + CHUNK - 1) / CHUNK;
  int64_t b1 = (nchunks + 7) / 8, b2 = (n + 7) / 8;
  const int64_t cap = (int64_t)kNumSMs * 16;
  segment_sum_phase1<DENSE><<<(int)(b1 > cap ? cap : b1), 256, 0, st>>>(w.keys_out, w.pos_out, w.seg_id, n, d, rows, dense,
                                                                       vocab, uniq_ids, uniq_rows, w.part);
  segment_sum_phase2<DENSE><<<(int)(b2 > cap ? cap : b2), 256, 0, st>>>(w.keys_out, w.seg_id, w.seg_start, n, d, dense,
                                                                       vocab, uniq_ids, uniq_rows, w.part);
  KGEB_LAUNCH_CHECK("segment_sum");
  return KGEB_OK;
}

static int sort_and_segment(const void* idx, int idx64, int64_t n, int64_t vocab, ScatterWs& w, int64_t* num_uniq,
                            cudaStream_t st, bool presorted = false) {
  const unsigned blocks = (unsigned)((n + 255) / 256);
  cudaError_t e;
  if (presorted) {  // keys already ascending: positions are the identity
    iota_keys_kernel<<<blocks, 256, 0, st>>>(idx, idx64, n, w.keys_out, w.pos_out);
  } else {
    iota_keys_kernel<<<blocks, 256, 0, st>>>(idx, idx64, n, w.keys_in, w.pos_in);
    int end_bit = 64;
    if (vocab > 0) {
      end_bit = 1;
      while (end_bit < 63 && ((int64_t)1 << end_bit) < vocab) ++end_bit;
    }
    e = cub::DeviceRadixSort::SortPairs(w.cub_tmp, w.cub_bytes, w.keys_in, w.keys_out, w.pos_in, w.pos_out, (int)n, 0,
                                        end_bit, st);
    if (e != cudaSuccess) return cuda_status(e, "radix sort");
  }
  head_flags_kernel<<<blocks, 256, 0, st>>>(w.keys_out, n, w.seg_id);
  e = cub::DeviceScan::InclusiveSum(w.cub_tmp, w.cub_bytes, w.seg_id, w.seg_id, (int)n, st);
  if (e != cudaSuccess) return cuda_status(e, "segment scan");
  seg_starts_kernel<<<blocks, 256, 0, st>>>(w.keys_out, w.seg_id, n, w.seg_start, num_uniq);
  KGEB_LAUNCH_CHECK("segment starts");
  return KGEB_OK;
}

// ------------------------------------------------------------------------------------------
// rows touched by the sparse gradient parts of an all-entity step (kgeb_touched_build / kgeb_touched_update)
// ------------------------------------------------------------------------------------------
constexpr int kTouchedThreads = 1024, kTouchedItems = 8, kTouchedMax = kTouchedThreads * kTouchedItems;

// One block: sort the <= 8192 ids, number the distinct in-shard ones 0.. in ascending order, publish slot_of[local id] and
// the slot of every input position (ids of other shards -> the dummy slot `dummy`).
__global__ void __launch_bounds__(kTouchedThreads, 1)
touched_build_kernel(const int64_t* __restrict__ ids_a, int n_a, const int64_t* __restrict__ ids_b, int n_b,
                     const int64_t* __restrict__ n_b_real, int64_t e_lo, int64_t e_hi, int32_t* __restrict__ slot_of,
                     int64_t* __restrict__ uniq, int64_t* __restrict__ num_uniq, int64_t* __restrict__ slot_a,
                     int64_t* __restrict__ slot_b, int64_t dummy) {
  using Sort = cub::BlockRadixSort<unsigned, kTouchedThreads, kTouchedItems>;
  using Scan = cub::BlockScan<int, kTouchedThreads>;
  __shared__ union { typename Sort::TempStorage sort; typename Scan::TempStorage scan; } tmp;
  __shared__ unsigned last_of[kTouchedThreads];
  const int t = threadIdx.x, n = n_a + n_b;
  // positions of ids_b past *n_b_real are padding: not touched; their slot is 0 (a sorted scatter whose permutation
  // places the padding first, as entity 0, still sees non-decreasing keys; padding entries carry zero rows)
  const int n_live = n_a + (n_b_real ? (int)min((int64_t)n_b, max((int64_t)0, *n_b_real)) : n_b);
  unsigned key[kTouchedItems];
#pragma unroll
  for (int j = 0; j < kTouchedItems; ++j) {
    const int i = t * kTouchedItems + j;
    unsigned k = 0xffffffffu;
    if (i < n_live) {
      const int64_t e = (i < n_a ? ids_a[i] : ids_b[i - n_a]);
      if (e >= e_lo && e < e_hi) k = (unsigned)(e - e_lo);
    }
    key[j] = k;
  }
  Sort(tmp.sort).Sort(key);        // blocked arrangement: thread t holds the sorted items [8 t, 8 t + 8)
  last_of[t] = key[kTouchedItems - 1];
  __syncthreads();
  const unsigned prev = t == 0 ? 0xffffffffu : last_of[t - 1];
  int heads = 0;
  bool head[kTouchedItems];
#pragma unroll
  for (int j = 0; j < kTouchedItems; ++j) {
    const unsigned before = j == 0 ? prev : key[j - 1];
    head[j] = key[j] != 0xffffffffu && (t * kTouchedItems + j == 0 || key[j] != before);
    heads += head[j];
  }
  int base, total;
  Scan(tmp.scan).ExclusiveSum(heads, base, total);
#pragma unroll
  for (int j = 0; j < kTouchedItems; ++j)
    if (head[j]) {
      slot_of[key[j]] = base;
      uniq[base] = (int64_t)key[j];
      ++base;
    }
  if (t == 0) *num_uniq = total;
  __threadfence_block();
  __syncthreads();
  for (int i = t; i < n; i += kTouchedThreads) {
    const int64_t e = (i < n_a ? ids_a[i] : ids_b[i - n_a]);
    const int64_t s = i >= n_live ? 0 : (e >= e_lo && e < e_hi) ? (int64_t)slot_of[e - e_lo] : dummy;
    if (i < n_a) slot_a[i] = s; else slot_b[i - n_a] = s;
  }
}

// Adagrad on the touched rows: gradient = dense part parked by the tile kernel + the summed sparse rows; clears the
// sparse buffer and the rows' slot_of entries for the next step.  skip != 0: clear only.
__global__ void touched_update_kernel(float* __restrict__ W, float* __restrict__ state, __nv_bfloat16* __restrict__ mirror,
                                      int32_t* __restrict__ slot_of, const int64_t* __restrict__ uniq,
                                      const int64_t* __restrict__ num_uniq, const float* __restrict__ g_dense,
                                      float* __restrict__ g_sparse, int64_t dummy, int d, float clr_val, float eps,
                                      const int* __restrict__ skip, const float* __restrict__ clr_dev) {
  const int64_t n = *num_uniq;
  const bool live = skip == nullptr || *skip == 0;
  const float clr = clr_dev ? *clr_dev : clr_val;   // the rate of this step from device memory (_sched entries)
  const int d4 = d / 4;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < (n + 1) * d4; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t slot = i / d4;
    const int c = (int)(i - slot * d4) * 4;
    if (slot == n) {      // the dummy row collects the rows of other shards
      *reinterpret_cast<float4*>(g_sparse + dummy * d + c) = make_float4(0.f, 0.f, 0.f, 0.f);
      continue;
    }
    const int64_t row = uniq[slot];
    float4* gs = reinterpret_cast<float4*>(g_sparse + slot * d + c);
    if (live) {
      float4 g = *reinterpret_cast<const float4*>(g_dense + slot * d + c);
      const float4 h = *gs;
      g.x += h.x; g.y += h.y; g.z += h.z; g.w += h.w;
      float4 w = *reinterpret_cast<float4*>(W + row * d + c), s = *reinterpret_cast<float4*>(state + row * d + c);
      s.x = fmaf(g.x, g.x, s.x); s.y = fmaf(g.y, g.y, s.y); s.z = fmaf(g.z, g.z, s.z); s.w = fmaf(g.w, g.w, s.w);
      w.x -= clr * g.x / (sqrtf(s.x) + eps);
      w.y -= clr * g.y / (sqrtf(s.y) + eps);
      w.z -= clr * g.z / (sqrtf(s.z) + eps);
      w.w -= clr * g.w / (sqrtf(s.w) + eps);
      *reinterpret_cast<float4*>(W + row * d + c) = w;
      *reinterpret_cast<float4*>(state + row * d + c) = s;
      if (mirror) {
        __nv_bfloat162 a = __floats2bfloat162_rn(w.x, w.y), b = __floats2bfloat162_rn(w.z, w.w);
        uint2 o;
        o.x = *reinterpret_cast<uint32_t*>(&a);
        o.y = *reinterpret_cast<uint32_t*>(&b);
        *reinterpret_cast<uint2*>(mirror + row * d + c) = o;
      }
    }
    *gs = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c == 0) slot_of[row] = -1;
  }
}

// ------------------------------------------------------------------------------------------
// optimizers
// ------------------------------------------------------------------------------------------
__global__ void adagrad_dense_kernel(float* __restrict__ W, float* __restrict__ state, const float* __restrict__ grad,
                                     const float* __restrict__ grad2, int64_t numel, float clr_val, float eps, float wd,
                                     __nv_bfloat16* __restrict__ mirror, const float* __restrict__ clr_dev) {
  const float clr = clr_dev ? *clr_dev : clr_val;   // the rate of this step from device memory (_sched entries)
  int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) * 4;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x * 4;
  for (; i + 3 < numel; i += stride) {
    float4 w = *reinterpret_cast<float4*>(W + i);
    float4 s = *reinterpret_cast<float4*>(state + i);
    float4 g = *reinterpret_cast<const float4*>(grad + i);
    if (grad2) {  // gradient accumulated in two buffers (dense / query-side parts written on different streams)
      const float4 h = *reinterpret_cast<const float4*>(grad2 + i);
      g.x += h.x; g.y += h.y; g.z += h.z; g.w += h.w;
    }
    g.x = fmaf(wd, w.x, g.x); g.y = fmaf(wd, w.y, g.y); g.z = fmaf(wd, w.z, g.z); g.w = fmaf(wd, w.w, g.w);
    s.x = fmaf(g.x, g.x, s.x); s.y = fmaf(g.y, g.y, s.y); s.z = fmaf(g.z, g.z, s.z); s.w = fmaf(g.w, g.w, s.w);
    w.x -= clr * g.x / (sqrtf(s.x) + eps);
    w.y -= clr * g.y / (sqrtf(s.y) + eps);
    w.z -= clr * g.z / (sqrtf(s.z) + eps);
    w.w -= clr * g.w / (sqrtf(s.w) + eps);
    *reinterpret_cast<float4*>(W + i) = w;
    *reinterpret_cast<float4*>(state + i) = s;
    if (mirror) {  // keep the bf16 mirror of the table in step with the fp32 master (KGEB_MATH_BF16)
      __nv_bfloat162 a = __floats2bfloat162_rn(w.x, w.y), b = __floats2bfloat162_rn(w.z, w.w);
      uint2 o;
      o.x = *reinterpret_cast<uint32_t*>(&a);
      o.y = *reinterpret_cast<uint32_t*>(&b);
      *reinterpret_cast<uint2*>(mirror + i) = o;
    }
  }
  // tail (numel % 4): handled by the thread whose i lands on it
  if (i < numel && i + 3 >= numel) {
    for (int64_t j = i; j < numel; ++j) {
      float g = fmaf(wd, W[j], grad[j] + (grad2 ? grad2[j] : 0.f));
      float s = fmaf(g, g, state[j]);
      state[j] = s;
      W[j] -= clr * g / (sqrtf(s) + eps);
      if (mirror) mirror[j] = __float2bfloat16_rn(W[j]);
    }
  }
}

__global__ void adagrad_rows_kernel(float* __restrict__ W, float* __restrict__ state, const int64_t* __restrict__ ids,
                                    const float* __restrict__ g, const int64_t* __restrict__ num_rows, int64_t max_rows,
                                    int d, float clr, float eps) {
  const int64_t nrows = min(*num_rows, max_rows);
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  for (; t < nrows * d; t += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = t / d;
    int c = (int)(t - r * d);
    int64_t dst = ids[r] * d + c;
    float gv = g[t];
    float s = fmaf(gv, gv, state[dst]);
    state[dst] = s;
    W[dst] -= clr * gv / (sqrtf(s) + eps);
  }
}

__global__ void adam_dense_kernel(float* __restrict__ W, float* __restrict__ m, float* __restrict__ v,
                                  const float* __restrict__ grad, int64_t numel, float lr, float b1, float b2, float eps,
                                  float wd, float bc1, float bc2) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const float step_size = lr / bc1;
  const float inv_sqrt_bc2 = rsqrtf(bc2);
  for (; i < numel; i += (int64_t)gridDim.x * blockDim.x) {
    float w = W[i];
    float g = fmaf(wd, w, grad[i]);
    float mi = m[i] + (1.f - b1) * (g - m[i]);  // lerp, as torch's exp_avg.lerp_(grad, 1-beta1)
    float vi = b2 * v[i] + (1.f - b2) * g * g;
    m[i] = mi;
    v[i] = vi;
    float denom = sqrtf(vi) * inv_sqrt_bc2 + eps;
    W[i] = w - step_size * (mi / denom);
  }
}

__global__ void csr_lookup_kernel(const int64_t* __restrict__ keys, int64_t nk, const int64_t* __restrict__ q,
                                  int64_t n, int64_t* __restrict__ out) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t a = q[2 * i], b = q[2 * i + 1];
  int64_t lo = 0, hi = nk;
  while (lo < hi) {  // lexicographic lower bound over [K,2]
    int64_t mid = (lo + hi) >> 1;
    int64_t ka = keys[2 * mid], kb = keys[2 * mid + 1];
    if (ka < a || (ka == a && kb < b)) lo = mid + 1; else hi = mid;
  }
  out[i] = (lo < nk && keys[2 * lo] == a && keys[2 * lo + 1] == b) ? lo : -1;
}

}  // namespace kgeb

using namespace kgeb;

extern "C" {

int64_t kgeb_scatter_workspace_bytes(int64_t n, int d) { return scatter_ws_bytes(n, d); }

int kgeb_scatter_add_rows(const void* idx, int idx64, const float* rows, int64_t n, int d, float* dense,
                          int64_t vocab, void* workspace, int64_t workspace_bytes, void* stream) {
  KGEB_REQUIRE(idx && rows && dense && n >= 0 && d > 0 && vocab > 0, "scatter_add_rows: bad arguments");
  KGEB_REQUIRE(n < ((int64_t)1 << 31), "scatter_add_rows: n too large");
  if (n == 0) return KGEB_OK;
  ScatterWs w;
  KGEB_REQUIRE(carve(workspace, workspace_bytes, n, d, w), "scatter_add_rows: workspace too small");
  cudaStream_t st = as_stream(stream);
  int rc = scatter_small(idx, idx64, rows, n, d, dense, vocab, w, st, false);
  if (rc >= 0) return rc;
  rc = sort_and_segment(idx, idx64, n, vocab, w, nullptr, st);
  if (rc) return rc;
  return segment_sums<true>(w, n, d, rows, dense, vocab, nullptr, nullptr, st);
}

int kgeb_scatter_add_rows_perm(const void* idx, int idx64, const int32_t* perm, const float* rows, int64_t n, int d,
                               float* dense, int64_t vocab, void* workspace, int64_t workspace_bytes, void* stream) {
  KGEB_REQUIRE(idx && perm && rows && dense && n >= 0 && d > 0 && vocab > 0, "scatter_add_rows_perm: bad arguments");
  if (n == 0) return KGEB_OK;
  const int pb = kgeb::bits_for(n), kb = kgeb::bits_for(vocab);
  KGEB_REQUIRE(n <= (1 << 26) && pb + kb <= 62, "scatter_add_rows_perm: n / vocab out of range");
  kgeb::ScatterWs w;
  KGEB_REQUIRE(kgeb::carve(workspace, workspace_bytes, n, d, w), "scatter_add_rows_perm: workspace too small");
  cudaStream_t st = as_stream(stream);
  const unsigned blocks = (unsigned)((n + 255) / 256);
  if (pb + kb > 32) {
    uint64_t* packed = reinterpret_cast<uint64_t*>(w.keys_in);
    kgeb::pack_perm_kernel<uint64_t><<<blocks, 256, 0, st>>>(idx, idx64, perm, (int)n, pb, packed);
    return kgeb::packed_phases<uint64_t>(packed, n, pb, d, rows, dense, vocab, w.part, st);
  }
  uint32_t* packed = reinterpret_cast<uint32_t*>(w.keys_in);
  kgeb::pack_perm_kernel<uint32_t><<<blocks, 256, 0, st>>>(idx, idx64, perm, (int)n, pb, packed);
  return kgeb::packed_phases<uint32_t>(packed, n, pb, d, rows, dense, vocab, w.part, st);
}

// internal: keys already ascending (e.g. label entries grouped by row)
int scatter_add_rows_presorted(const int64_t* keys, const float* rows, int64_t n, int d, float* dense, int64_t vocab,
                               void* workspace, int64_t workspace_bytes, cudaStream_t st) {
  if (n == 0) return KGEB_OK;
  kgeb::ScatterWs w;
  KGEB_REQUIRE(kgeb::carve(workspace, workspace_bytes, n, d, w), "scatter_add_rows(presorted): workspace too small");
  int rc = kgeb::scatter_small(keys, 1, rows, n, d, dense, vocab, w, st, true);
  if (rc >= 0) return rc;
  rc = kgeb::sort_and_segment(keys, 1, n, vocab, w, nullptr, st, true);
  if (rc) return rc;
  return kgeb::segment_sums<true>(w, n, d, rows, dense, vocab, nullptr, nullptr, st);
}

int kgeb_segment_reduce_rows(const void* idx, int idx64, const float* rows, int64_t n, int d, int64_t* uniq_ids,
                             float* uniq_rows, int64_t* num_uniq, void* workspace, int64_t workspace_bytes,
                             void* stream) {
  KGEB_REQUIRE(idx && rows && uniq_ids && uniq_rows && num_uniq && n >= 0 && d > 0, "segment_reduce_rows: bad arguments");
  KGEB_REQUIRE(n < ((int64_t)1 << 31), "segment_reduce_rows: n too large");
  cudaStream_t st = as_stream(stream);
  if (n == 0) {
    cudaMemsetAsync(num_uniq, 0, sizeof(int64_t), st);
    return KGEB_OK;
  }
  ScatterWs w;
  KGEB_REQUIRE(carve(workspace, workspace_bytes, n, d, w), "segment_reduce_rows: workspace too small");
  int rc = sort_and_segment(idx, idx64, n, 0, w, num_uniq, st);
  if (rc) return rc;
  return segment_sums<false>(w, n, d, rows, nullptr, 0, uniq_ids, uniq_rows, st);
}

int kgeb_touched_capacity(void) { return kgeb::kTouchedMax; }

int kgeb_touched_build(const int64_t* ids_a, int64_t n_a, const int64_t* ids_b, int64_t n_b, const int64_t* n_b_real,
                       int64_t e_lo, int64_t e_hi, int32_t* slot_of, int64_t* uniq_rows, int64_t* num_uniq, int64_t* slot_a,
                       int64_t* slot_b, void* stream) {
  KGEB_REQUIRE(n_a >= 0 && n_b >= 0 && n_a + n_b <= kgeb::kTouchedMax, "touched_build: at most %d ids per step (got %lld)",
               kgeb::kTouchedMax, (long long)(n_a + n_b));
  KGEB_REQUIRE((n_a == 0 || (ids_a && slot_a)) && (n_b == 0 || (ids_b && slot_b)) && slot_of && uniq_rows && num_uniq &&
                   e_hi >= e_lo && e_hi - e_lo < ((int64_t)1 << 32) - 1,
               "touched_build: bad arguments");
  kgeb::touched_build_kernel<<<1, kgeb::kTouchedThreads, 0, as_stream(stream)>>>(
      ids_a, (int)n_a, ids_b, (int)n_b, n_b_real, e_lo, e_hi, slot_of, uniq_rows, num_uniq, slot_a, slot_b, n_a + n_b);
  KGEB_LAUNCH_CHECK("touched_build");
  return KGEB_OK;
}

}  // extern "C"

// The by-value entries and their _sched siblings (rate read from a device word) share one kernel each: clr_dev == NULL
// selects the by-value rate.
static int touched_update(float* W, float* state, void* bf16_mirror, int32_t* slot_of, const int64_t* uniq_rows,
                          const int64_t* num_uniq, int64_t capacity, const float* g_dense, float* g_sparse, int d, float clr,
                          const float* clr_dev, float eps, const int32_t* skip_flag, void* stream) {
  KGEB_REQUIRE(W && state && slot_of && uniq_rows && num_uniq && g_dense && g_sparse && capacity > 0 && d > 0 && d % 4 == 0,
               "touched_update: bad arguments");
  const int64_t work = (capacity + 1) * (d / 4);
  int64_t blocks = (work + 255) / 256;
  if (blocks > (int64_t)kNumSMs * 8) blocks = (int64_t)kNumSMs * 8;
  kgeb::touched_update_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(
      W, state, reinterpret_cast<__nv_bfloat16*>(bf16_mirror), slot_of, uniq_rows, num_uniq, g_dense, g_sparse, capacity, d,
      clr, eps, skip_flag, clr_dev);
  KGEB_LAUNCH_CHECK("touched_update");
  return KGEB_OK;
}

static int adagrad_dense(float* W, float* state, const float* grad, const float* grad2, int64_t numel, float clr,
                         const float* clr_dev, float eps, float weight_decay, void* bf16_mirror, void* stream) {
  KGEB_REQUIRE(W && state && grad && numel >= 0, "adagrad_dense: bad arguments");
  KGEB_REQUIRE(((reinterpret_cast<uintptr_t>(W) | reinterpret_cast<uintptr_t>(state) |
                 reinterpret_cast<uintptr_t>(grad) | reinterpret_cast<uintptr_t>(grad2)) & 15) == 0,
               "adagrad_dense: pointers must be 16-byte aligned");
  if (numel == 0) return KGEB_OK;
  int64_t blocks = (numel / 4 + 255) / 256 + 1;
  int grid = (int)(blocks > (int64_t)kNumSMs * 8 ? (int64_t)kNumSMs * 8 : blocks);
  adagrad_dense_kernel<<<grid, 256, 0, as_stream(stream)>>>(W, state, grad, grad2, numel, clr, eps, weight_decay,
                                                            reinterpret_cast<__nv_bfloat16*>(bf16_mirror), clr_dev);
  KGEB_LAUNCH_CHECK("adagrad_dense");
  return KGEB_OK;
}

extern "C" {

int kgeb_touched_update(float* W, float* state, void* bf16_mirror, int32_t* slot_of, const int64_t* uniq_rows,
                        const int64_t* num_uniq, int64_t capacity, const float* g_dense, float* g_sparse, int d, float clr,
                        float eps, const int32_t* skip_flag, void* stream) {
  return touched_update(W, state, bf16_mirror, slot_of, uniq_rows, num_uniq, capacity, g_dense, g_sparse, d, clr, nullptr,
                        eps, skip_flag, stream);
}

int kgeb_touched_update_sched(float* W, float* state, void* bf16_mirror, int32_t* slot_of, const int64_t* uniq_rows,
                              const int64_t* num_uniq, int64_t capacity, const float* g_dense, float* g_sparse, int d,
                              const float* clr, float eps, const int32_t* skip_flag, void* stream) {
  KGEB_REQUIRE(clr, "touched_update_sched: the learning-rate word is NULL");
  return touched_update(W, state, bf16_mirror, slot_of, uniq_rows, num_uniq, capacity, g_dense, g_sparse, d, 0.f, clr, eps,
                        skip_flag, stream);
}

int kgeb_adagrad_dense(float* W, float* state, const float* grad, const float* grad2, int64_t numel, float clr,
                       float eps, float weight_decay, void* bf16_mirror, void* stream) {
  return adagrad_dense(W, state, grad, grad2, numel, clr, nullptr, eps, weight_decay, bf16_mirror, stream);
}

int kgeb_adagrad_dense_sched(float* W, float* state, const float* grad, const float* grad2, int64_t numel, const float* clr,
                             float eps, float weight_decay, void* bf16_mirror, void* stream) {
  KGEB_REQUIRE(clr, "adagrad_dense_sched: the learning-rate word is NULL");
  return adagrad_dense(W, state, grad, grad2, numel, 0.f, clr, eps, weight_decay, bf16_mirror, stream);
}

int kgeb_adagrad_rows(float* W, float* state, const int64_t* row_ids, const float* row_grads,
                      const int64_t* num_rows_dev, int64_t max_rows, int d, float clr, float eps, void* stream) {
  KGEB_REQUIRE(W && state && row_ids && row_grads && num_rows_dev && max_rows >= 0 && d > 0, "adagrad_rows: bad arguments");
  if (max_rows == 0) return KGEB_OK;
  int64_t blocks = (max_rows * d + 255) / 256;
  int grid = (int)(blocks > (int64_t)kNumSMs * 8 ? (int64_t)kNumSMs * 8 : blocks);
  adagrad_rows_kernel<<<grid, 256, 0, as_stream(stream)>>>(W, state, row_ids, row_grads, num_rows_dev, max_rows, d, clr, eps);
  KGEB_LAUNCH_CHECK("adagrad_rows");
  return KGEB_OK;
}

int kgeb_adam_dense(float* W, float* exp_avg, float* exp_avg_sq, const float* grad, int64_t numel, float lr,
                    float beta1, float beta2, float eps, float weight_decay, float bias_corr1, float bias_corr2,
                    void* stream) {
  KGEB_REQUIRE(W && exp_avg && exp_avg_sq && grad && numel >= 0, "adam_dense: bad arguments");
  if (numel == 0) return KGEB_OK;
  int64_t blocks = (numel + 255) / 256;
  int grid = (int)(blocks > (int64_t)kNumSMs * 8 ? (int64_t)kNumSMs * 8 : blocks);
  adam_dense_kernel<<<grid, 256, 0, as_stream(stream)>>>(W, exp_avg, exp_avg_sq, grad, numel, lr, beta1, beta2, eps,
                                                         weight_decay, bias_corr1, bias_corr2);
  KGEB_LAUNCH_CHECK("adam_dense");
  return KGEB_OK;
}

int kgeb_csr_lookup(const int64_t* keys, int64_t num_keys, const int64_t* query_pairs, int64_t n, int64_t* row_out,
                    void* stream) {
  KGEB_REQUIRE(keys && query_pairs && row_out && num_keys >= 0 && n >= 0, "csr_lookup: bad arguments");
  if (n == 0) return KGEB_OK;
  csr_lookup_kernel<<<(unsigned)((n + 255) / 256), 256, 0, as_stream(stream)>>>(keys, num_keys, query_pairs, n, row_out);
  KGEB_LAUNCH_CHECK("csr_lookup");
  return KGEB_OK;
}

}  // extern "C"
