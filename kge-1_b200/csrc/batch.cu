// On-device batch construction from device-resident KvsAllIndex arrays (SURVEY.md 8f-1): the steps *before* the hot
// path that the reference does with Python dict lookups per triple.
//   * filter CSR of an evaluation batch   -- EntityRankingJob._collate + get_sp_po_coords_from_spo_batch
//     (kge/job/entity_ranking.py:53-77, kge/job/util.py:5-38)
//   * query rows + label CSR of a KvsAll training batch -- TrainingJobKvsAll collate (kge/job/train.py:590-677)
// Both are "gather CSR rows": a count pass (one thread per source list: key binary search, length), an exclusive
// scan by the caller, and a fill pass (one warp per source list, coalesced copies).  Integer work only; results are
// bit-exact by construction and compared against the reference's coordinates in the tests.
#include <cstdint>

#include <cub/cub.cuh>

#include "common.cuh"

namespace kgeb {

constexpr int MAX_SPLITS = 4;

struct IndexSet {            // K splits x (sp index, po index), passed by value to the kernels
  kgeb_index_t sp[MAX_SPLITS];
  kgeb_index_t po[MAX_SPLITS];
  int k;
};

// row of the key pair (a, b) in the lexicographically sorted keys [num_keys, 2], or -1
__device__ __forceinline__ int64_t find_key(const kgeb_index_t& ix, int64_t a, int64_t b) {
  int64_t lo = 0, hi = ix.num_keys;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    const int64_t ka = ix.keys[2 * mid], kb = ix.keys[2 * mid + 1];
    if (ka < a || (ka == a && kb < b)) lo = mid + 1; else hi = mid;
  }
  return (lo < ix.num_keys && ix.keys[2 * lo] == a && ix.keys[2 * lo + 1] == b) ? lo : -1;
}

// Source list j = row * K + k of an evaluation batch: rows [0,B) = known objects of (s,p) in split k, rows [B,2B) =
// known subjects of (p,o) in split k.
__global__ void filter_count_kernel(IndexSet set, const void* __restrict__ s, const void* __restrict__ p,
                                    const void* __restrict__ o, int idx64, int64_t B, int64_t* __restrict__ src_row,
                                    int64_t* __restrict__ len) {
  const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j >= 2 * B * set.k) return;
  const int64_t row = j / set.k;
  const int k = (int)(j % set.k);
  const bool sp = row < B;
  const int64_t t = sp ? row : row - B;
  const kgeb_index_t& ix = sp ? set.sp[k] : set.po[k];
  const int64_t a = sp ? load_index(s, idx64, t) : load_index(p, idx64, t);
  const int64_t b = sp ? load_index(p, idx64, t) : load_index(o, idx64, t);
  const int64_t r = find_key(ix, a, b);
  src_row[j] = r;
  len[j] = r < 0 ? 0 : ix.offsets[r + 1] - ix.offsets[r];
}

// one warp per source list: values -> col[pos[j] ...]; key_out (optional) = (row << 32) | value for the per-row sort
__global__ void __launch_bounds__(256)
filter_fill_kernel(IndexSet set, int64_t B, const int64_t* __restrict__ src_row, const int64_t* __restrict__ pos,
                   int64_t* __restrict__ col, int64_t* __restrict__ key_out) {
  const int lane = threadIdx.x & 31;
  const int64_t j = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (j >= 2 * B * set.k) return;
  const int64_t r = src_row[j];
  if (r < 0) return;
  const int64_t row = j / set.k;
  const int k = (int)(j % set.k);
  const kgeb_index_t& ix = row < B ? set.sp[k] : set.po[k];
  const int64_t b0 = ix.offsets[r], n = ix.offsets[r + 1] - b0, dst = pos[j];
  for (int64_t i = lane; i < n; i += 32) {
    const int64_t v = ix.values[b0 + i];
    if (col) col[dst + i] = v;
    if (key_out) key_out[dst + i] = (row << 32) | v;
  }
}

// KvsAll training batch: example id < n_sp is the sp-query with key row id of the sp index, the others are po-queries
// (train.py:611-640: queries = the key pair, labels = the values of that key).
// inv_rel_offset = R > 0 (reciprocal relations model, reciprocal_relations_model.py:70-83): a po-query (p, o) becomes the
// sp-query (o, p + R) with the same labels.
__global__ void kvsall_count_kernel(kgeb_index_t sp, kgeb_index_t po, const int64_t* __restrict__ ids, int64_t B,
                                    int64_t inv_rel_offset, int64_t* __restrict__ a_idx, int64_t* __restrict__ p_idx,
                                    int32_t* __restrict__ row_combine, int64_t* __restrict__ len) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= B) return;
  const int64_t id = ids[i];
  const bool is_sp = id < sp.num_keys;
  const kgeb_index_t& ix = is_sp ? sp : po;
  const int64_t r = is_sp ? id : id - sp.num_keys;
  // sp key = (s, p): entity first; po key = (p, o): entity second
  a_idx[i] = is_sp ? ix.keys[2 * r] : ix.keys[2 * r + 1];
  p_idx[i] = is_sp ? ix.keys[2 * r + 1] : ix.keys[2 * r] + inv_rel_offset;
  row_combine[i] = (is_sp || inv_rel_offset > 0) ? KGEB_SP_ : KGEB__PO;
  len[i] = ix.offsets[r + 1] - ix.offsets[r];
}

__global__ void __launch_bounds__(256)
kvsall_fill_kernel(kgeb_index_t sp, kgeb_index_t po, const int64_t* __restrict__ ids, int64_t B,
                   const int64_t* __restrict__ lab_off, int64_t capacity, int64_t* __restrict__ lab_col,
                   int32_t* __restrict__ overflow) {
  const int lane = threadIdx.x & 31;
  const int64_t i = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (i >= B) return;
  const int64_t id = ids[i];
  const bool is_sp = id < sp.num_keys;
  const kgeb_index_t& ix = is_sp ? sp : po;
  const int64_t r = is_sp ? id : id - sp.num_keys;
  const int64_t b0 = ix.offsets[r], n = ix.offsets[r + 1] - b0, dst = lab_off[i];
  if (dst + n > capacity) {          // the static label buffer of the graph-captured step is too small for this batch
    if (lane == 0) *overflow = 1;
    return;
  }
  for (int64_t k = lane; k < n; k += 32) lab_col[dst + k] = ix.values[b0 + k];
}

__global__ void iota_kernel(int32_t* __restrict__ out, int64_t n, int64_t* __restrict__ first_off) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) out[i] = (int32_t)i;
  if (i == 0 && first_off) *first_off = 0;
}

static int bits_needed(int64_t x) {  // smallest b with 2^b >= x
  int b = 1;
  while (b < 62 && ((int64_t)1 << b) < x) ++b;
  return b;
}
static size_t up256(size_t x) { return (x + 255) / 256 * 256; }

struct BuildWs {
  int64_t* keys_tmp;   // [n] sorted keys (discarded)
  int32_t* iota;       // [n]
  void* cub_tmp;
  size_t cub_bytes;
};
static size_t build_cub_bytes(int64_t n) {
  size_t a = 0, b = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, a, (const int64_t*)nullptr, (int64_t*)nullptr, (const int32_t*)nullptr,
                                  (int32_t*)nullptr, (int)n, 0, 40);
  cub::DeviceScan::InclusiveSum(nullptr, b, (const int64_t*)nullptr, (int64_t*)nullptr, (int)n);
  return a > b ? a : b;
}

// ------------------------------------------------------------------------------------------
// 1vsAll batch (train.py:1032-1062) straight from the [B, 3] triples: the static inputs of the captured step and the
// three stable argsorts, one block, no host work.  Rows 0..B-1 are the sp_ queries (label = o), rows B..2B-1 the _po
// queries (label = s); every row has exactly one label.  inv_rel_offset = R > 0: rows B..2B-1 are the sp_ queries (o, p + R)
// of a reciprocal relations model instead (label = s).
// ------------------------------------------------------------------------------------------
constexpr int kOvaThreads = 1024, kOvaItems = 8, kOvaMax = kOvaThreads * kOvaItems;   // 2 B <= 8192

__global__ void __launch_bounds__(kOvaThreads, 1)
onevsall_build_kernel(const int64_t* __restrict__ triples, int B, int64_t inv_rel_offset, int64_t* __restrict__ a_idx,
                      int64_t* __restrict__ p_idx,
                      int32_t* __restrict__ row_combine, int64_t* __restrict__ lab_off, int64_t* __restrict__ lab_col,
                      int32_t* __restrict__ a_perm, int32_t* __restrict__ p_perm, int32_t* __restrict__ lab_perm) {
  using Sort = cub::BlockRadixSort<unsigned, kOvaThreads, kOvaItems, int>;
  __shared__ typename Sort::TempStorage tmp;
  const int t = threadIdx.x, n = 2 * B;
  for (int i = t; i < n; i += kOvaThreads) {
    const int r = i < B ? i : i - B;
    const int64_t s = triples[3 * r], p = triples[3 * r + 1], o = triples[3 * r + 2];
    a_idx[i] = i < B ? s : o;
    p_idx[i] = i < B ? p : p + inv_rel_offset;
    lab_col[i] = i < B ? o : s;
    row_combine[i] = (i < B || inv_rel_offset > 0) ? 0 : 1;
    lab_off[i] = i;
  }
  if (t == 0) lab_off[n] = n;
  // stable argsort of each id list (LSD radix sort keeps the order of equal keys; padding keys sort last)
  for (int which = 0; which < 3; ++which) {
    unsigned key[kOvaItems];
    int val[kOvaItems];
#pragma unroll
    for (int j = 0; j < kOvaItems; ++j) {
      const int i = t * kOvaItems + j;
      unsigned k = 0xffffffffu;
      if (i < n) {
        const int r = i < B ? i : i - B;
        const int col = which == 1 ? 1 : ((which == 0) == (i < B) ? 0 : 2);   // a: s | o ;  p: p | p ;  labels: o | s
        k = (unsigned)triples[3 * r + col];
        if (which == 1 && i >= B) k += (unsigned)inv_rel_offset;
      }
      key[j] = k;
      val[j] = i;
    }
    __syncthreads();
    Sort(tmp).Sort(key, val);
    int32_t* out = which == 0 ? a_perm : (which == 1 ? p_perm : lab_perm);
#pragma unroll
    for (int j = 0; j < kOvaItems; ++j) {
      const int i = t * kOvaItems + j;
      if (i < n) out[i] = val[j];
    }
  }
}

static bool index_ok(const kgeb_index_t& ix) { return ix.num_keys >= 0 && (ix.num_keys == 0 || (ix.keys && ix.offsets && ix.values)); }

}  // namespace kgeb

using namespace kgeb;

extern "C" {

int kgeb_filter_csr_count(const kgeb_index_t* sp_indexes, const kgeb_index_t* po_indexes, int num_splits, const void* s,
                          const void* p, const void* o, int idx64, int64_t B, int64_t* src_row, int64_t* len,
                          void* stream) {
  KGEB_REQUIRE(num_splits >= 1 && num_splits <= MAX_SPLITS, "filter_csr: 1..%d splits (got %d)", MAX_SPLITS, num_splits);
  KGEB_REQUIRE(sp_indexes && po_indexes && s && p && o && src_row && len && B >= 0, "filter_csr_count: bad arguments");
  if (B == 0) return KGEB_OK;
  IndexSet set;
  set.k = num_splits;
  for (int k = 0; k < num_splits; ++k) {
    KGEB_REQUIRE(index_ok(sp_indexes[k]) && index_ok(po_indexes[k]), "filter_csr_count: index %d has NULL arrays", k);
    set.sp[k] = sp_indexes[k];
    set.po[k] = po_indexes[k];
  }
  const int64_t n = 2 * B * num_splits;
  filter_count_kernel<<<(unsigned)((n + 127) / 128), 128, 0, as_stream(stream)>>>(set, s, p, o, idx64, B, src_row, len);
  KGEB_LAUNCH_CHECK("filter_count");
  return KGEB_OK;
}

int kgeb_filter_csr_fill(const kgeb_index_t* sp_indexes, const kgeb_index_t* po_indexes, int num_splits, int64_t B,
                         const int64_t* src_row, const int64_t* pos, int64_t* col, int64_t* sort_keys, void* stream) {
  KGEB_REQUIRE(num_splits >= 1 && num_splits <= MAX_SPLITS, "filter_csr: 1..%d splits (got %d)", MAX_SPLITS, num_splits);
  KGEB_REQUIRE(sp_indexes && po_indexes && src_row && pos && (col || sort_keys) && B >= 0, "filter_csr_fill: bad arguments");
  if (B == 0) return KGEB_OK;
  IndexSet set;
  set.k = num_splits;
  for (int k = 0; k < num_splits; ++k) {
    set.sp[k] = sp_indexes[k];
    set.po[k] = po_indexes[k];
  }
  const int64_t n = 2 * B * num_splits;
  filter_fill_kernel<<<(unsigned)((n + 7) / 8), 256, 0, as_stream(stream)>>>(set, B, src_row, pos, col, sort_keys);
  KGEB_LAUNCH_CHECK("filter_fill");
  return KGEB_OK;
}

int kgeb_kvsall_batch_count(const kgeb_index_t* sp_index, const kgeb_index_t* po_index, const int64_t* example_ids,
                            int64_t B, int64_t* a_idx, int64_t* p_idx, int32_t* row_combine, int64_t* len, void* stream) {
  KGEB_REQUIRE(sp_index && po_index && example_ids && a_idx && p_idx && row_combine && len && B >= 0,
               "kvsall_batch_count: bad arguments");
  KGEB_REQUIRE(index_ok(*sp_index) && index_ok(*po_index), "kvsall_batch_count: index has NULL arrays");
  if (B == 0) return KGEB_OK;
  kvsall_count_kernel<<<(unsigned)((B + 127) / 128), 128, 0, as_stream(stream)>>>(*sp_index, *po_index, example_ids, B, 0,
                                                                                 a_idx, p_idx, row_combine, len);
  KGEB_LAUNCH_CHECK("kvsall_count");
  return KGEB_OK;
}

int kgeb_kvsall_batch_fill(const kgeb_index_t* sp_index, const kgeb_index_t* po_index, const int64_t* example_ids,
                           int64_t B, const int64_t* lab_off, int64_t capacity, int64_t* lab_col, int32_t* overflow,
                           void* stream) {
  KGEB_REQUIRE(sp_index && po_index && example_ids && lab_off && lab_col && overflow && B >= 0 && capacity >= 0,
               "kvsall_batch_fill: bad arguments");
  if (B == 0) return KGEB_OK;
  kvsall_fill_kernel<<<(unsigned)((B + 7) / 8), 256, 0, as_stream(stream)>>>(*sp_index, *po_index, example_ids, B,
                                                                             lab_off, capacity, lab_col, overflow);
  KGEB_LAUNCH_CHECK("kvsall_fill");
  return KGEB_OK;
}

int64_t kgeb_kvsall_build_workspace_bytes(int64_t B, int64_t capacity) {
  const int64_t n = (B > capacity ? B : capacity) + 1;
  return (int64_t)(up256((size_t)n * 8) + up256((size_t)n * 4) + up256(build_cub_bytes(n)) + 1024);
}

int kgeb_kvsall_batch_build_inv(const kgeb_index_t* sp_index, const kgeb_index_t* po_index, const int64_t* example_ids,
                                int64_t B, int64_t capacity, int64_t num_entities, int64_t num_relations, int64_t* a_idx,
                                int64_t* p_idx, int32_t* row_combine, int64_t* lab_off, int64_t* lab_col, int32_t* a_perm,
                                int32_t* p_perm, int32_t* lab_perm, int32_t* overflow, void* workspace,
                                int64_t workspace_bytes, int64_t inv_rel_offset, void* stream) {
  KGEB_REQUIRE(sp_index && po_index && example_ids && a_idx && p_idx && row_combine && lab_off && lab_col && a_perm &&
                   p_perm && lab_perm && overflow && workspace,
               "kvsall_batch_build: NULL argument");
  KGEB_REQUIRE(B > 0 && capacity > 0 && B < ((int64_t)1 << 30) && capacity < ((int64_t)1 << 30),
               "kvsall_batch_build: batch size / label capacity out of range");
  KGEB_REQUIRE(index_ok(*sp_index) && index_ok(*po_index), "kvsall_batch_build: index has NULL arrays");
  KGEB_REQUIRE(workspace_bytes >= kgeb_kvsall_build_workspace_bytes(B, capacity), "kvsall_batch_build: workspace too small");
  KGEB_REQUIRE(inv_rel_offset >= 0, "kvsall_batch_build: negative inverse relation offset");
  cudaStream_t st = as_stream(stream);
  const int64_t n = (B > capacity ? B : capacity) + 1;
  char* wp = reinterpret_cast<char*>(workspace);
  BuildWs w;
  w.keys_tmp = reinterpret_cast<int64_t*>(wp);  wp += up256((size_t)n * 8);
  w.iota = reinterpret_cast<int32_t*>(wp);      wp += up256((size_t)n * 4);
  w.cub_tmp = wp;
  w.cub_bytes = build_cub_bytes(n);
  cudaError_t e;
  iota_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(w.iota, n, lab_off);
  kvsall_count_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(*sp_index, *po_index, example_ids, B, inv_rel_offset,
                                                                  a_idx, p_idx, row_combine, lab_off + 1);
  KGEB_LAUNCH_CHECK("kvsall_count");
  size_t bytes = w.cub_bytes;
  e = cub::DeviceScan::InclusiveSum(w.cub_tmp, bytes, lab_off + 1, lab_off + 1, (int)B, st);
  if (e != cudaSuccess) return cuda_status(e, "kvsall_batch_build scan");
  e = cudaMemsetAsync(lab_col, 0, (size_t)capacity * 8, st);   // padding counts as entity 0 in lab_perm
  if (e == cudaSuccess) e = cudaMemsetAsync(overflow, 0, 4, st);
  if (e != cudaSuccess) return cuda_status(e, "kvsall_batch_build memset");
  kvsall_fill_kernel<<<(unsigned)((B + 7) / 8), 256, 0, st>>>(*sp_index, *po_index, example_ids, B, lab_off, capacity,
                                                             lab_col, overflow);
  KGEB_LAUNCH_CHECK("kvsall_fill");
  // the three stable argsorts (ids of the batch are known here, so the step's scatters need no sort)
  const int eb = bits_needed(num_entities), rb = bits_needed(num_relations + inv_rel_offset);
  bytes = w.cub_bytes;
  e = cub::DeviceRadixSort::SortPairs(w.cub_tmp, bytes, (const int64_t*)a_idx, w.keys_tmp, (const int32_t*)w.iota, a_perm,
                                      (int)B, 0, eb, st);
  bytes = w.cub_bytes;
  if (e == cudaSuccess)
    e = cub::DeviceRadixSort::SortPairs(w.cub_tmp, bytes, (const int64_t*)p_idx, w.keys_tmp, (const int32_t*)w.iota, p_perm,
                                        (int)B, 0, rb, st);
  bytes = w.cub_bytes;
  if (e == cudaSuccess)
    e = cub::DeviceRadixSort::SortPairs(w.cub_tmp, bytes, (const int64_t*)lab_col, w.keys_tmp, (const int32_t*)w.iota,
                                        lab_perm, (int)capacity, 0, eb, st);
  if (e != cudaSuccess) return cuda_status(e, "kvsall_batch_build sort");
  return KGEB_OK;
}

int kgeb_kvsall_batch_build(const kgeb_index_t* sp_index, const kgeb_index_t* po_index, const int64_t* example_ids,
                            int64_t B, int64_t capacity, int64_t num_entities, int64_t num_relations, int64_t* a_idx,
                            int64_t* p_idx, int32_t* row_combine, int64_t* lab_off, int64_t* lab_col, int32_t* a_perm,
                            int32_t* p_perm, int32_t* lab_perm, int32_t* overflow, void* workspace,
                            int64_t workspace_bytes, void* stream) {
  return kgeb_kvsall_batch_build_inv(sp_index, po_index, example_ids, B, capacity, num_entities, num_relations, a_idx, p_idx,
                                     row_combine, lab_off, lab_col, a_perm, p_perm, lab_perm, overflow, workspace,
                                     workspace_bytes, 0, stream);
}

int kgeb_onevsall_batch_build_inv(const int64_t* triples, int64_t B, int64_t num_entities, int64_t num_relations,
                                  int64_t* a_idx, int64_t* p_idx, int32_t* row_combine, int64_t* lab_off, int64_t* lab_col,
                                  int32_t* a_perm, int32_t* p_perm, int32_t* lab_perm, int64_t inv_rel_offset, void* stream) {
  KGEB_REQUIRE(triples && a_idx && p_idx && row_combine && lab_off && lab_col && a_perm && p_perm && lab_perm,
               "onevsall_batch_build: NULL buffer");
  KGEB_REQUIRE(B >= 1 && 2 * B <= kgeb::kOvaMax, "onevsall_batch_build: 1 <= batch <= %d (got %lld)", kgeb::kOvaMax / 2,
               (long long)B);
  KGEB_REQUIRE(inv_rel_offset >= 0, "onevsall_batch_build: negative inverse relation offset");
  KGEB_REQUIRE(num_entities < ((int64_t)1 << 32) - 1 && num_relations + inv_rel_offset < ((int64_t)1 << 32) - 1,
               "onevsall_batch_build: ids must fit 32 bits");
  kgeb::onevsall_build_kernel<<<1, kgeb::kOvaThreads, 0, as_stream(stream)>>>(triples, (int)B, inv_rel_offset, a_idx, p_idx,
                                                                             row_combine, lab_off, lab_col, a_perm, p_perm,
                                                                             lab_perm);
  KGEB_LAUNCH_CHECK("onevsall_batch_build");
  return KGEB_OK;
}

int kgeb_onevsall_batch_build(const int64_t* triples, int64_t B, int64_t num_entities, int64_t num_relations, int64_t* a_idx,
                              int64_t* p_idx, int32_t* row_combine, int64_t* lab_off, int64_t* lab_col, int32_t* a_perm,
                              int32_t* p_perm, int32_t* lab_perm, void* stream) {
  return kgeb_onevsall_batch_build_inv(triples, B, num_entities, num_relations, a_idx, p_idx, row_combine, lab_off, lab_col,
                                       a_perm, p_perm, lab_perm, 0, stream);
}

}  // extern "C"
