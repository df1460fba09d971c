// Lp penalties of LookupEmbedder fused with their gradient and with the row update (SURVEY.md 8f-3).
//   reference: LookupEmbedder.penalty (kge/model/embedder/lookup_embedder.py:112-158), summed per embedder by
//   KgeModel.penalty (kge/model/kge_model.py:588-606); each term is back-propagated on its own between the loss
//   backward and optimizer.step() (kge/job/train.py:320-338).
//     unweighted: value = w/p * sum |W|^p                       d value / dW = w * |W|^(p-1) * sign(W)      (whole table)
//     weighted:   value = w/p * sum_u c_u * sum_k |W[u,k]|^p / n   over the distinct indexes u of the batch with
//                 multiplicities c_u, n = number of indexes     d value / dW[u,:] = w * c_u / n * |W[u,:]|^(p-1) * sign
//   All of it is HBM-bound elementwise work: the dense form costs one extra pass over the table in the reference (plus
//   the autograd pass back); here the dense gradient term is formed inside the Adagrad kernel from the parameter value
//   it reads anyway (kgeb_adagrad_dense_lp: 0 extra bytes) and the penalty value is a by-product of the same pass.
//   Values are reduced in a fixed order (per-block partials, then one block): deterministic.
#include <cstdint>

#include <cub/cub.cuh>
#include <cuda_bf16.h>

#include "common.cuh"

namespace kgeb {

// |x|^p and d/dx (|x|^p / p) = |x|^(p-1) sign(x) for integer p >= 1
__device__ __forceinline__ void lp_terms(float x, int p, float& pw, float& dv) {
  const float a = fabsf(x);
  if (p == 2) { pw = x * x; dv = x; return; }
  if (p == 1) { pw = a; dv = sgnf(x); return; }
  if (p == 3) { pw = a * a * a; dv = x * a; return; }
  float m = 1.f;                       // a^(p-1)
  for (int k = 1; k < p; ++k) m *= a;
  pw = m * a;
  dv = m * sgnf(x);
}

constexpr int kPenBlock = 256;

__device__ __forceinline__ float block_sum_fixed(float v, float* sh) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) sh[w] = v;
  __syncthreads();
  float t = 0.f;
  if (threadIdx.x == 0)
    for (int k = 0; k < (int)(blockDim.x >> 5); ++k) t += sh[k];
  return t;   // valid in thread 0
}

__global__ void __launch_bounds__(kPenBlock)
lp_dense_kernel(const float* __restrict__ W, int64_t numel, int p, float weight, float* __restrict__ grad,
                float* __restrict__ partial) {
  __shared__ float sh[kPenBlock / 32];
  float acc = 0.f;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < numel; i += (int64_t)gridDim.x * blockDim.x) {
    float pw, dv;
    lp_terms(W[i], p, pw, dv);
    acc += pw;
    if (grad) grad[i] = fmaf(weight, dv, grad[i]);
  }
  const float t = block_sum_fixed(acc, sh);
  if (threadIdx.x == 0) partial[blockIdx.x] = t;
}

// value_out[0] = scale * sum partial[0..n) in index order (one block; double accumulation)
__global__ void __launch_bounds__(256)
finish_value_kernel(const float* __restrict__ partial, const int64_t* __restrict__ n_dev, int64_t n, float scale,
                    float* __restrict__ value_out) {
  __shared__ double sh[256];
  if (n_dev) n = min(n, *n_dev);
  // contiguous slices per thread, combined in thread order: fixed association for a given n
  const int64_t per = (n + 255) / 256;
  const int64_t lo = min(n, (int64_t)threadIdx.x * per), hi = min(n, lo + per);
  double a = 0.0;
  for (int64_t i = lo; i < hi; ++i) a += (double)partial[i];
  sh[threadIdx.x] = a;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int k = 0; k < 256; ++k) t += sh[k];
    value_out[0] = (float)(t * (double)scale);
  }
}

// Adagrad step (torch.optim.Adagrad; clr = lr / (1 + (step - 1) * lr_decay) from the caller) with the unweighted Lp penalty
// folded in:
//   g = grad (+ grad2) + weight_decay * w + pen_weight * |w|^(p-1) sign(w);  state += g^2;  w -= clr * g / (sqrt(state) + eps)
// and the block partial sums of |w|^p of the *pre-update* parameters (the penalty value the reference reports).
__global__ void __launch_bounds__(kPenBlock)
adagrad_dense_lp_kernel(float* __restrict__ W, float* __restrict__ state, const float* __restrict__ grad,
                        const float* __restrict__ grad2, int64_t numel, float clr_val, float eps, float wd, int p,
                        float pen_weight, __nv_bfloat16* __restrict__ mirror, float* __restrict__ partial,
                        const float* __restrict__ clr_dev) {
  __shared__ float sh[kPenBlock / 32];
  const float clr = clr_dev ? *clr_dev : clr_val;   // the rate of this step from device memory (_sched entry)
  float acc = 0.f;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < numel; i += (int64_t)gridDim.x * blockDim.x) {
    const float w = W[i];
    float pw, dv;
    lp_terms(w, p, pw, dv);
    acc += pw;
    float g = grad[i] + (grad2 ? grad2[i] : 0.f);
    g = fmaf(wd, w, g);
    g = fmaf(pen_weight, dv, g);
    const float s = fmaf(g, g, state[i]);
    state[i] = s;
    const float wn = w - clr * g / (sqrtf(s) + eps);
    W[i] = wn;
    if (mirror) mirror[i] = __float2bfloat16_rn(wn);
  }
  const float t = block_sum_fixed(acc, sh);
  if (threadIdx.x == 0) partial[blockIdx.x] = t;
}

// weighted form: one warp per distinct index (run of the sorted index list)
__global__ void __launch_bounds__(256)
lp_rows_kernel(const float* __restrict__ W, int64_t vocab, int dim, const int64_t* __restrict__ uniq,
               const int32_t* __restrict__ counts, const int64_t* __restrict__ num_runs, int64_t max_runs, int p,
               float weight, float inv_n, float* __restrict__ grad, float* __restrict__ partial) {
  const int lane = threadIdx.x & 31;
  const int64_t run = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (run >= max_runs) return;
  float acc = 0.f;
  if (run < *num_runs) {
    const int64_t u = uniq[run];
    const float c = (float)counts[run];
    if (u >= 0 && u < vocab) {
      for (int k = lane; k < dim; k += 32) {
        float pw, dv;
        lp_terms(W[u * dim + k], p, pw, dv);
        acc += pw * c;
        if (grad) grad[u * dim + k] = fmaf(weight * c * inv_n, dv, grad[u * dim + k]);
      }
    }
  }
  acc = warp_sum(acc);
  if (lane == 0) partial[run] = acc;   // 0 for the unused tail: the finish kernel may sum all max_runs entries
}

__global__ void widen_index_kernel(const void* __restrict__ idx, int idx64, int64_t n, int64_t* __restrict__ out) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) out[i] = load_index(idx, idx64, i);
}

static inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }
static inline int dense_grid(int64_t numel) {
  const int64_t blocks = (numel + kPenBlock - 1) / kPenBlock;
  return (int)(blocks > (int64_t)kNumSMs * 8 ? (int64_t)kNumSMs * 8 : (blocks < 1 ? 1 : blocks));
}

struct RowsLayout {
  size_t keys_in, keys_out, uniq, counts, num_runs, partial, cub, cub_bytes, total;
};
static RowsLayout rows_layout(int64_t n) {
  RowsLayout l;
  size_t sort_bytes = 0, rle_bytes = 0;
  cub::DeviceRadixSort::SortKeys(nullptr, sort_bytes, (const int64_t*)nullptr, (int64_t*)nullptr, (int)n);
  cub::DeviceRunLengthEncode::Encode(nullptr, rle_bytes, (const int64_t*)nullptr, (int64_t*)nullptr, (int32_t*)nullptr,
                                     (int64_t*)nullptr, (int)n);
  size_t o = 0;
  l.keys_in = o; o += align256((size_t)n * 8);
  l.keys_out = o; o += align256((size_t)n * 8);
  l.uniq = o; o += align256((size_t)n * 8);
  l.counts = o; o += align256((size_t)n * 4);
  l.num_runs = o; o += 256;
  l.partial = o; o += align256((size_t)n * 4);
  l.cub = o;
  l.cub_bytes = sort_bytes > rle_bytes ? sort_bytes : rle_bytes;
  o += align256(l.cub_bytes);
  l.total = o;
  return l;
}

}  // namespace kgeb

using namespace kgeb;

extern "C" {

int64_t kgeb_penalty_workspace_bytes(int64_t n_indexes, int64_t numel) {
  if (n_indexes < 0 || numel < 0 || n_indexes >= ((int64_t)1 << 31)) return -1;
  const size_t dense = align256((size_t)dense_grid(numel) * 4);
  const size_t rows = n_indexes > 0 ? rows_layout(n_indexes).total : 0;
  return (int64_t)(dense > rows ? dense : rows) + 256;
}

int kgeb_lp_penalty_dense(const float* W, int64_t numel, int p, float weight, float* grad, float* value_out,
                          void* workspace, int64_t workspace_bytes, void* stream) {
  KGEB_REQUIRE(W && value_out && workspace && numel >= 0, "lp_penalty_dense: bad arguments");
  KGEB_REQUIRE(p >= 1 && p <= 16, "lp_penalty_dense: p = %d not in [1, 16]", p);
  const int grid = dense_grid(numel);
  KGEB_REQUIRE(workspace_bytes >= (int64_t)grid * 4, "lp_penalty_dense: workspace too small");
  float* partial = reinterpret_cast<float*>(workspace);
  lp_dense_kernel<<<grid, kPenBlock, 0, as_stream(stream)>>>(W, numel, p, weight, grad, partial);
  KGEB_LAUNCH_CHECK("lp_dense");
  finish_value_kernel<<<1, 256, 0, as_stream(stream)>>>(partial, nullptr, grid, weight / (float)p, value_out);
  KGEB_LAUNCH_CHECK("lp_finish");
  return KGEB_OK;
}

int kgeb_lp_penalty_rows(const float* W, int64_t vocab, int dim, const void* indexes, int idx64, int64_t n, int p,
                         float weight, float* grad, float* value_out, void* workspace, int64_t workspace_bytes,
                         void* stream) {
  KGEB_REQUIRE(W && indexes && value_out && workspace && vocab > 0 && dim > 0 && n > 0 && n < ((int64_t)1 << 31),
               "lp_penalty_rows: bad arguments");
  KGEB_REQUIRE(p >= 1 && p <= 16, "lp_penalty_rows: p = %d not in [1, 16]", p);
  const RowsLayout l = rows_layout(n);
  KGEB_REQUIRE(workspace_bytes >= (int64_t)l.total, "lp_penalty_rows: workspace too small (%lld < %lld)",
               (long long)workspace_bytes, (long long)l.total);
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  int64_t* keys_in = reinterpret_cast<int64_t*>(ws + l.keys_in);
  int64_t* keys_out = reinterpret_cast<int64_t*>(ws + l.keys_out);
  int64_t* uniq = reinterpret_cast<int64_t*>(ws + l.uniq);
  int32_t* counts = reinterpret_cast<int32_t*>(ws + l.counts);
  int64_t* num_runs = reinterpret_cast<int64_t*>(ws + l.num_runs);
  float* partial = reinterpret_cast<float*>(ws + l.partial);
  cudaStream_t st = as_stream(stream);
  widen_index_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(indexes, idx64, n, keys_in);
  KGEB_LAUNCH_CHECK("lp_rows widen");
  size_t cub_bytes = l.cub_bytes;
  int bits = 1;
  while (bits < 63 && ((int64_t)1 << bits) < vocab) ++bits;
  cudaError_t e = cub::DeviceRadixSort::SortKeys(ws + l.cub, cub_bytes, keys_in, keys_out, (int)n, 0, bits, st);
  if (e != cudaSuccess) return cuda_status(e, "lp_rows sort");
  cub_bytes = l.cub_bytes;
  e = cub::DeviceRunLengthEncode::Encode(ws + l.cub, cub_bytes, keys_out, uniq, counts, num_runs, (int)n, st);
  if (e != cudaSuccess) return cuda_status(e, "lp_rows run-length encode");
  lp_rows_kernel<<<(unsigned)((n + 7) / 8), 256, 0, st>>>(W, vocab, dim, uniq, counts, num_runs, n, p, weight,
                                                         1.f / (float)n, grad, partial);
  KGEB_LAUNCH_CHECK("lp_rows");
  finish_value_kernel<<<1, 256, 0, st>>>(partial, nullptr, n, weight / (float)p / (float)n, value_out);
  KGEB_LAUNCH_CHECK("lp_rows finish");
  return KGEB_OK;
}

}  // extern "C"

// kgeb_adagrad_dense_lp and its _sched sibling: one kernel, clr_dev == NULL selects the by-value rate
static int adagrad_dense_lp(float* W, float* state, const float* grad, const float* grad2, int64_t numel, float clr,
                            const float* clr_dev, float eps, float weight_decay, int p, float pen_weight, void* bf16_mirror,
                            float* value_out, void* workspace, int64_t workspace_bytes, void* stream) {
  KGEB_REQUIRE(W && state && grad && value_out && workspace && numel >= 0, "adagrad_dense_lp: bad arguments");
  KGEB_REQUIRE(p >= 1 && p <= 16, "adagrad_dense_lp: p = %d not in [1, 16]", p);
  const int grid = dense_grid(numel);
  KGEB_REQUIRE(workspace_bytes >= (int64_t)grid * 4, "adagrad_dense_lp: workspace too small");
  float* partial = reinterpret_cast<float*>(workspace);
  adagrad_dense_lp_kernel<<<grid, kPenBlock, 0, as_stream(stream)>>>(W, state, grad, grad2, numel, clr, eps, weight_decay, p,
                                                                    pen_weight, reinterpret_cast<__nv_bfloat16*>(bf16_mirror),
                                                                    partial, clr_dev);
  KGEB_LAUNCH_CHECK("adagrad_dense_lp");
  finish_value_kernel<<<1, 256, 0, as_stream(stream)>>>(partial, nullptr, grid, pen_weight / (float)p, value_out);
  KGEB_LAUNCH_CHECK("adagrad_dense_lp finish");
  return KGEB_OK;
}

extern "C" {

int kgeb_adagrad_dense_lp(float* W, float* state, const float* grad, const float* grad2, int64_t numel, float clr,
                          float eps, float weight_decay, int p, float pen_weight, void* bf16_mirror, float* value_out,
                          void* workspace, int64_t workspace_bytes, void* stream) {
  return adagrad_dense_lp(W, state, grad, grad2, numel, clr, nullptr, eps, weight_decay, p, pen_weight, bf16_mirror,
                          value_out, workspace, workspace_bytes, stream);
}

int kgeb_adagrad_dense_lp_sched(float* W, float* state, const float* grad, const float* grad2, int64_t numel,
                                const float* clr, float eps, float weight_decay, int p, float pen_weight, void* bf16_mirror,
                                float* value_out, void* workspace, int64_t workspace_bytes, void* stream) {
  KGEB_REQUIRE(clr, "adagrad_dense_lp_sched: the learning-rate word is NULL");
  return adagrad_dense_lp(W, state, grad, grad2, numel, 0.f, clr, eps, weight_decay, p, pen_weight, bf16_mirror, value_out,
                          workspace, workspace_bytes, stream);
}

}  // extern "C"
