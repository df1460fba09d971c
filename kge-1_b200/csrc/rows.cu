// Row-wise (HBM/L2-bound) kernels: gather, "spo" scoring of the seven scorers and its backward,
// query transforms of the sp_/_po forms, and negative-sampling pair scoring.
// One warp per row; lanes stride the embedding dimension so every load is a coalesced 128 B line
// (float4 per lane where the row is 16 B aligned).  Reference call sites are cited in kgeb200.h.
#include "common.cuh"
#include <stdarg.h>
#include <string.h>

namespace kgeb {

static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int cuda_status(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return KGEB_OK;
  set_error("%s: %s", what, cudaGetErrorString(e));
  return KGEB_ERR_CUDA;
}

constexpr int kWarpsPerBlock = 8;
constexpr float kPairwiseEps = 1e-6f;  // torch.nn.functional.pairwise_distance default eps

__device__ __forceinline__ int relation_dim(int model, int d) {
  return (model == KGEB_CP || model == KGEB_ROTATE) ? d / 2 : (model == KGEB_RESCAL ? d * d : d);
}

// ------------------------------------------------------------------------------------------
// gather
// ------------------------------------------------------------------------------------------
__global__ void gather_rows_v4(const float4* __restrict__ W, int64_t vocab, int dim4, const void* idx,
                               int idx64, int64_t n, float4* __restrict__ out) {
  // one thread per float4; consecutive threads cover one row then the next -> coalesced stores
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int64_t total = n * dim4;
  for (; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = t / dim4;
    int c = (int)(t - r * dim4);
    int64_t src = load_index(idx, idx64, r);
    out[t] = __ldg(&W[src * dim4 + c]);
  }
}
// rows of an entity-sharded table: W holds the rows [e_lo, e_hi) of the global table; ids outside give zero rows (the
// owners' partial results are summed by an all-reduce).  local_ids (optional) = id - e_lo, or e_hi - e_lo for "not mine".
__global__ void gather_rows_shard_kernel(const float* __restrict__ W, int64_t e_lo, int64_t e_hi, int dim,
                                         const void* idx, int idx64, int64_t n, float* __restrict__ out,
                                         int64_t* __restrict__ local_ids) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t total = n * dim;
  for (; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = t / dim;
    const int c = (int)(t - r * dim);
    const int64_t e = load_index(idx, idx64, r);
    const bool mine = e >= e_lo && e < e_hi;
    out[t] = mine ? __ldg(&W[(e - e_lo) * dim + c]) : 0.f;
    if (c == 0 && local_ids) local_ids[r] = mine ? e - e_lo : e_hi - e_lo;
  }
}
__global__ void gather_rows_v1(const float* __restrict__ W, int64_t vocab, int dim, const void* idx,
                               int idx64, int64_t n, float* __restrict__ out) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int64_t total = n * dim;
  for (; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = t / dim;
    int c = (int)(t - r * dim);
    out[t] = __ldg(&W[load_index(idx, idx64, r) * dim + c]);
  }
}

// ------------------------------------------------------------------------------------------
// spo forward: warp per triple
// ------------------------------------------------------------------------------------------
struct RowSrc {
  const float* base;
  const void* idx;
};
__device__ __forceinline__ const float* row_ptr(const float* base, const void* idx, int idx64, int64_t i,
                                                int width) {
  return base + load_index(idx, idx64, i) * (int64_t)width;
}

template <int MODEL>
__device__ __forceinline__ float spo_row(const float* __restrict__ s, const float* __restrict__ p,
                                         const float* __restrict__ o, int d, int l_norm, int lane) {
  const int h = d >> 1;
  float acc = 0.f;
  if (MODEL == KGEB_DISTMULT) {
    for (int k = lane; k < d; k += 32) acc += s[k] * p[k] * o[k];
  } else if (MODEL == KGEB_COMPLEX) {
    for (int k = lane; k < h; k += 32) {
      float sr = s[k], si = s[k + h], pr = p[k], pi = p[k + h], orr = o[k], oi = o[k + h];
      acc += sr * pr * orr + si * pr * oi + sr * pi * oi - si * pi * orr;
    }
  } else if (MODEL == KGEB_CP) {
    for (int k = lane; k < h; k += 32) acc += s[k] * p[k] * o[k + h];
  } else if (MODEL == KGEB_SIMPLE) {
    for (int k = lane; k < h; k += 32) acc += s[k] * p[k] * o[k + h] + s[k + h] * p[k + h] * o[k];
    acc *= 0.5f;
  } else if (MODEL == KGEB_RESCAL) {
    for (int i = 0; i < d; ++i) {
      float si = s[i];
      const float* mrow = p + (int64_t)i * d;
      for (int j = lane; j < d; j += 32) acc += si * mrow[j] * o[j];
    }
  } else if (MODEL == KGEB_TRANSE) {
    for (int k = lane; k < d; k += 32) {
      float df = s[k] + p[k] - o[k] + kPairwiseEps;
      acc += (l_norm == 1) ? fabsf(df) : df * df;
    }
  } else if (MODEL == KGEB_ROTATE) {
    for (int k = lane; k < h; k += 32) {
      float pr, pi;
      sincosf(p[k], &pi, &pr);
      float sr = s[k], si = s[k + h];
      float re = sr * pr - si * pi - o[k];
      float im = sr * pi + si * pr - o[k + h];
      float m2 = re * re + im * im;
      acc += (l_norm == 1) ? sqrtf(m2) : m2;
    }
  }
  acc = warp_sum(acc);
  if (MODEL == KGEB_TRANSE) acc = (l_norm == 1) ? -acc : -sqrtf(acc);
  if (MODEL == KGEB_ROTATE) acc = (l_norm == 1) ? acc : sqrtf(acc);
  return acc;
}

template <int MODEL>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
score_spo_kernel(int l_norm, const float* s_src, const void* s_idx, const float* p_src, const void* p_idx,
                 const float* o_src, const void* o_idx, int idx64, int64_t n, int d, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  int64_t row = blockIdx.x * (int64_t)kWarpsPerBlock + (threadIdx.x >> 5);
  const int dr = relation_dim(MODEL, d);
  for (; row < n; row += (int64_t)gridDim.x * kWarpsPerBlock) {
    const float* s = row_ptr(s_src, s_idx, idx64, row, d);
    const float* p = row_ptr(p_src, p_idx, idx64, row, dr);
    const float* o = row_ptr(o_src, o_idx, idx64, row, d);
    float v = spo_row<MODEL>(s, p, o, d, l_norm, lane);
    if (lane == 0) out[row] = v;
  }
}

// ------------------------------------------------------------------------------------------
// spo backward: warp per triple, per-row gradients (dense [n,*]); scattering is a separate step
// ------------------------------------------------------------------------------------------
template <int MODEL>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
score_spo_bwd_kernel(int l_norm, const float* s_src, const void* s_idx, const float* p_src, const void* p_idx,
                     const float* o_src, const void* o_idx, int idx64, int64_t n, int d,
                     const float* __restrict__ gout, float* __restrict__ ds, float* __restrict__ dp,
                     float* __restrict__ d_o) {
  const int lane = threadIdx.x & 31;
  const int h = d >> 1;
  const int dr = relation_dim(MODEL, d);
  int64_t row = blockIdx.x * (int64_t)kWarpsPerBlock + (threadIdx.x >> 5);
  for (; row < n; row += (int64_t)gridDim.x * kWarpsPerBlock) {
    const float* s = row_ptr(s_src, s_idx, idx64, row, d);
    const float* p = row_ptr(p_src, p_idx, idx64, row, dr);
    const float* o = row_ptr(o_src, o_idx, idx64, row, d);
    float* gs = ds + row * d;
    float* gp = dp + row * (int64_t)dr;
    float* go = d_o + row * d;
    const float g = gout[row];
    if (MODEL == KGEB_DISTMULT) {
      for (int k = lane; k < d; k += 32) {
        float a = s[k], b = p[k], c = o[k];
        gs[k] = g * b * c;
        gp[k] = g * a * c;
        go[k] = g * a * b;
      }
    } else if (MODEL == KGEB_COMPLEX) {
      for (int k = lane; k < h; k += 32) {
        float sr = s[k], si = s[k + h], pr = p[k], pi = p[k + h], orr = o[k], oi = o[k + h];
        gs[k] = g * (pr * orr + pi * oi);
        gs[k + h] = g * (pr * oi - pi * orr);
        gp[k] = g * (sr * orr + si * oi);
        gp[k + h] = g * (sr * oi - si * orr);
        go[k] = g * (sr * pr - si * pi);
        go[k + h] = g * (si * pr + sr * pi);
      }
    } else if (MODEL == KGEB_CP) {
      for (int k = lane; k < h; k += 32) {
        float a = s[k], b = p[k], c = o[k + h];
        gs[k] = g * b * c;
        gs[k + h] = 0.f;
        gp[k] = g * a * c;
        go[k + h] = g * a * b;
        go[k] = 0.f;
      }
    } else if (MODEL == KGEB_SIMPLE) {
      const float gh = 0.5f * g;
      for (int k = lane; k < h; k += 32) {
        float sh = s[k], st = s[k + h], pf = p[k], pb = p[k + h], oh = o[k], ot = o[k + h];
        gs[k] = gh * pf * ot;
        gs[k + h] = gh * pb * oh;
        gp[k] = gh * sh * ot;
        gp[k + h] = gh * st * oh;
        go[k + h] = gh * sh * pf;
        go[k] = gh * st * pb;
      }
    } else if (MODEL == KGEB_RESCAL) {
      // ds_i = g sum_j M_ij o_j ; do_j = g sum_i s_i M_ij ; dM_ij = g s_i o_j
      for (int j = lane; j < d; j += 32) go[j] = 0.f;
      __syncwarp();
      for (int i = 0; i < d; ++i) {
        const float* mrow = p + (int64_t)i * d;
        float si = s[i];
        float acc = 0.f;
        for (int j = lane; j < d; j += 32) {
          float m = mrow[j], oj = o[j];
          acc += m * oj;
          go[j] += g * si * m;  // lane-private columns j = lane (mod 32)
          gp[(int64_t)i * d + j] = g * si * oj;
        }
        acc = warp_sum(acc);
        if (lane == 0) gs[i] = g * acc;
      }
    } else if (MODEL == KGEB_TRANSE) {
      float acc = 0.f;
      if (l_norm != 1) {
        for (int k = lane; k < d; k += 32) {
          float df = s[k] + p[k] - o[k] + kPairwiseEps;
          acc += df * df;
        }
        acc = sqrtf(warp_sum(acc));
      }
      const float inv = (l_norm == 1 || acc == 0.f) ? 0.f : 1.f / acc;
      for (int k = lane; k < d; k += 32) {
        float df = s[k] + p[k] - o[k] + kPairwiseEps;
        float dd = (l_norm == 1) ? -sgnf(df) : -df * inv;  // d score / d diff
        gs[k] = g * dd;
        gp[k] = g * dd;
        go[k] = -g * dd;
      }
    } else if (MODEL == KGEB_ROTATE) {
      float acc = 0.f;
      if (l_norm != 1) {
        for (int k = lane; k < h; k += 32) {
          float pr, pi;
          sincosf(p[k], &pi, &pr);
          float re = s[k] * pr - s[k + h] * pi - o[k];
          float im = s[k] * pi + s[k + h] * pr - o[k + h];
          acc += re * re + im * im;
        }
        acc = sqrtf(warp_sum(acc));
      }
      for (int k = lane; k < h; k += 32) {
        float pr, pi;
        sincosf(p[k], &pi, &pr);
        float sr = s[k], si = s[k + h];
        float re = sr * pr - si * pi - o[k];
        float im = sr * pi + si * pr - o[k + h];
        float den = (l_norm == 1) ? sqrtf(re * re + im * im) : acc;
        float inv = den == 0.f ? 0.f : 1.f / den;
        float dre = g * re * inv, dim_ = g * im * inv;
        gs[k] = dre * pr + dim_ * pi;
        gs[k + h] = -dre * pi + dim_ * pr;
        go[k] = -dre;
        go[k + h] = -dim_;
        gp[k] = dre * (-sr * pi - si * pr) + dim_ * (sr * pr - si * pi);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// query transforms (SURVEY.md Appendix D)
// ------------------------------------------------------------------------------------------
template <int MODEL>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
query_build_kernel(int combine, const int32_t* __restrict__ row_combine, const float* a_src, const void* a_idx,
                   const float* p_src, const void* p_idx, int idx64, int64_t n, int d, float* __restrict__ Q) {
  const int lane = threadIdx.x & 31;
  const int h = d >> 1;
  const int dr = relation_dim(MODEL, d);
  int64_t row = blockIdx.x * (int64_t)kWarpsPerBlock + (threadIdx.x >> 5);
  for (; row < n; row += (int64_t)gridDim.x * kWarpsPerBlock) {
    const bool sp = ((row_combine ? row_combine[row] : combine) == KGEB_SP_);
    const float* a = row_ptr(a_src, a_idx, idx64, row, d);
    const float* p = row_ptr(p_src, p_idx, idx64, row, dr);
    float* q = Q + row * d;
    if (MODEL == KGEB_DISTMULT) {
      for (int k = lane; k < d; k += 32) q[k] = a[k] * p[k];
    } else if (MODEL == KGEB_COMPLEX) {
      for (int k = lane; k < h; k += 32) {
        float ar = a[k], ai = a[k + h], pr = p[k], pi = p[k + h];
        if (sp) {
          q[k] = ar * pr - ai * pi;
          q[k + h] = ai * pr + ar * pi;
        } else {
          q[k] = pr * ar + pi * ai;
          q[k + h] = pr * ai - pi * ar;
        }
      }
    } else if (MODEL == KGEB_CP) {
      for (int k = lane; k < h; k += 32) {
        if (sp) {  // candidates contribute o[:, h:]
          q[k] = 0.f;
          q[k + h] = a[k] * p[k];
        } else {  // candidates contribute s[:, :h]
          q[k] = a[k + h] * p[k];
          q[k + h] = 0.f;
        }
      }
    } else if (MODEL == KGEB_SIMPLE) {
      for (int k = lane; k < h; k += 32) {
        float ah = a[k], at = a[k + h], pf = p[k], pb = p[k + h];
        if (sp) {  // 1/2 [s_t*p_b | s_h*p_f]
          q[k] = 0.5f * (at * pb);
          q[k + h] = 0.5f * (ah * pf);
        } else {  // 1/2 [o_t*p_f | o_h*p_b]
          q[k] = 0.5f * (at * pf);
          q[k + h] = 0.5f * (ah * pb);
        }
      }
    } else if (MODEL == KGEB_RESCAL) {
      if (sp) {  // q_j = sum_i s_i M_ij : lanes over j, coalesced rows of M
        for (int j = lane; j < d; j += 32) {
          float acc = 0.f;
          for (int i = 0; i < d; ++i) acc += a[i] * p[(int64_t)i * d + j];
          q[j] = acc;
        }
      } else {  // q_i = sum_j M_ij o_j
        for (int i = 0; i < d; ++i) {
          float acc = 0.f;
          for (int j = lane; j < d; j += 32) acc += p[(int64_t)i * d + j] * a[j];
          acc = warp_sum(acc);
          if (lane == 0) q[i] = acc;
        }
      }
    } else if (MODEL == KGEB_TRANSE) {
      for (int k = lane; k < d; k += 32) q[k] = sp ? a[k] + p[k] : a[k] - p[k];
    } else if (MODEL == KGEB_ROTATE) {
      for (int k = lane; k < h; k += 32) {
        float pr, pi;
        sincosf(p[k], &pi, &pr);
        float ar = a[k], ai = a[k + h];
        if (sp) {  // s * r
          q[k] = ar * pr - ai * pi;
          q[k + h] = ar * pi + ai * pr;
        } else {  // o * conj(r)
          q[k] = ar * pr + ai * pi;
          q[k + h] = ai * pr - ar * pi;
        }
      }
    }
  }
}

template <int MODEL>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
query_bwd_kernel(int combine, const int32_t* __restrict__ row_combine, const float* a_src, const void* a_idx,
                 const float* p_src, const void* p_idx, int idx64, int64_t n, int d, const float* __restrict__ dQ,
                 float* __restrict__ da, float* __restrict__ dp) {
  const int lane = threadIdx.x & 31;
  const int h = d >> 1;
  const int dr = relation_dim(MODEL, d);
  int64_t row = blockIdx.x * (int64_t)kWarpsPerBlock + (threadIdx.x >> 5);
  for (; row < n; row += (int64_t)gridDim.x * kWarpsPerBlock) {
    const bool sp = ((row_combine ? row_combine[row] : combine) == KGEB_SP_);
    const float* a = row_ptr(a_src, a_idx, idx64, row, d);
    const float* p = row_ptr(p_src, p_idx, idx64, row, dr);
    const float* g = dQ + row * d;
    float* ga = da + row * d;
    float* gp = dp + row * (int64_t)dr;
    if (MODEL == KGEB_DISTMULT) {
      for (int k = lane; k < d; k += 32) {
        ga[k] = g[k] * p[k];
        gp[k] = g[k] * a[k];
      }
    } else if (MODEL == KGEB_COMPLEX) {
      for (int k = lane; k < h; k += 32) {
        float ar = a[k], ai = a[k + h], pr = p[k], pi = p[k + h], gr = g[k], gi = g[k + h];
        if (sp) {
          ga[k] = gr * pr + gi * pi;
          ga[k + h] = -gr * pi + gi * pr;
          gp[k] = gr * ar + gi * ai;
          gp[k + h] = -gr * ai + gi * ar;
        } else {
          ga[k] = gr * pr - gi * pi;
          ga[k + h] = gr * pi + gi * pr;
          gp[k] = gr * ar + gi * ai;
          gp[k + h] = gr * ai - gi * ar;
        }
      }
    } else if (MODEL == KGEB_CP) {
      for (int k = lane; k < h; k += 32) {
        if (sp) {
          ga[k] = g[k + h] * p[k];
          ga[k + h] = 0.f;
          gp[k] = g[k + h] * a[k];
        } else {
          ga[k + h] = g[k] * p[k];
          ga[k] = 0.f;
          gp[k] = g[k] * a[k + h];
        }
      }
    } else if (MODEL == KGEB_SIMPLE) {
      for (int k = lane; k < h; k += 32) {
        float ah = a[k], at = a[k + h], pf = p[k], pb = p[k + h];
        float g0 = 0.5f * g[k], g1 = 0.5f * g[k + h];
        if (sp) {  // q0 = at*pb, q1 = ah*pf
          ga[k + h] = g0 * pb;
          gp[k + h] = g0 * at;
          ga[k] = g1 * pf;
          gp[k] = g1 * ah;
        } else {  // q0 = at*pf, q1 = ah*pb
          ga[k + h] = g0 * pf;
          gp[k] = g0 * at;
          ga[k] = g1 * pb;
          gp[k + h] = g1 * ah;
        }
      }
    } else if (MODEL == KGEB_RESCAL) {
      if (sp) {  // q_j = sum_i s_i M_ij : ds_i = sum_j M_ij g_j ; dM_ij = s_i g_j
        for (int i = 0; i < d; ++i) {
          float acc = 0.f, ai = a[i];
          for (int j = lane; j < d; j += 32) {
            float gj = g[j];
            acc += p[(int64_t)i * d + j] * gj;
            gp[(int64_t)i * d + j] = ai * gj;
          }
          acc = warp_sum(acc);
          if (lane == 0) ga[i] = acc;
        }
      } else {  // q_i = sum_j M_ij o_j : do_j = sum_i M_ij g_i ; dM_ij = g_i o_j
        for (int j = lane; j < d; j += 32) {
          float acc = 0.f, oj = a[j];
          for (int i = 0; i < d; ++i) {
            float gi = g[i];
            acc += p[(int64_t)i * d + j] * gi;
            gp[(int64_t)i * d + j] = gi * oj;
          }
          ga[j] = acc;
        }
      }
    } else if (MODEL == KGEB_TRANSE) {
      for (int k = lane; k < d; k += 32) {
        ga[k] = g[k];
        gp[k] = sp ? g[k] : -g[k];
      }
    } else if (MODEL == KGEB_ROTATE) {
      for (int k = lane; k < h; k += 32) {
        float pr, pi;
        sincosf(p[k], &pi, &pr);
        float ar = a[k], ai = a[k + h], gr = g[k], gi = g[k + h];
        if (sp) {  // q_re = ar pr - ai pi ; q_im = ar pi + ai pr
          ga[k] = gr * pr + gi * pi;
          ga[k + h] = -gr * pi + gi * pr;
          gp[k] = gr * (-ar * pi - ai * pr) + gi * (ar * pr - ai * pi);
        } else {  // q_re = ar pr + ai pi ; q_im = ai pr - ar pi
          ga[k] = gr * pr - gi * pi;
          ga[k + h] = gr * pi + gi * pr;
          gp[k] = gr * (-ar * pi + ai * pr) + gi * (-ai * pi - ar * pr);
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// negative-sampling pair scoring: warp per (row, candidate); the query row is read from L1/L2
// ------------------------------------------------------------------------------------------
template <int KIND>
__device__ __forceinline__ float pair_accumulate_nosum(const float* __restrict__ q, const float* __restrict__ c,
                                                       int d, int lane) {
  float acc = 0.f;
  if (KIND == KGEB_ROT_L1) {
    const int h = d >> 1;
    for (int k = lane; k < h; k += 32) {
      float re = q[k] - c[k], im = q[k + h] - c[k + h];
      acc += sqrtf(re * re + im * im);
    }
  } else if ((d & 3) == 0) {
    const float4* q4 = reinterpret_cast<const float4*>(q);
    const float4* c4 = reinterpret_cast<const float4*>(c);
    for (int k = lane; k < (d >> 2); k += 32) {
      float4 a = q4[k], b = __ldg(&c4[k]);
      if (KIND == KGEB_DOT) {
        acc += a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w;
      } else if (KIND == KGEB_NEG_L1) {
        acc += fabsf(a.x - b.x) + fabsf(a.y - b.y) + fabsf(a.z - b.z) + fabsf(a.w - b.w);
      } else {
        float x = a.x - b.x, y = a.y - b.y, z = a.z - b.z, w = a.w - b.w;
        acc += x * x + y * y + z * z + w * w;
      }
    }
  } else {
    for (int k = lane; k < d; k += 32) {
      float x = q[k] - c[k];
      acc += (KIND == KGEB_DOT) ? q[k] * c[k] : (KIND == KGEB_NEG_L1 ? fabsf(x) : x * x);
    }
  }
  return acc;      // this lane's part: warp_sum() of it is the pair's sum
}
template <int KIND>
__device__ __forceinline__ float pair_accumulate(const float* __restrict__ q, const float* __restrict__ c, int d, int lane) {
  return warp_sum(pair_accumulate_nosum<KIND>(q, c, d, lane));
}
template <int KIND>
__device__ __forceinline__ float pair_finish(float acc) {
  if (KIND == KGEB_NEG_L1) return -acc;
  if (KIND == KGEB_NEG_L2) return -sqrtf(acc);
  if (KIND == KGEB_ROT_L2) return sqrtf(acc);
  return acc;
}

template <int KIND>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
pairs_score_kernel(const float* __restrict__ Q, const float* __restrict__ table, const void* cand, int idx64,
                   int64_t B, int64_t M, int d, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  int64_t pair = blockIdx.x * (int64_t)kWarpsPerBlock + (threadIdx.x >> 5);
  const int64_t total = B * M;
  for (; pair < total; pair += (int64_t)gridDim.x * kWarpsPerBlock) {
    int64_t row = pair / M;
    const float* q = Q + row * d;
    const float* c = table + load_index(cand, idx64, pair) * (int64_t)d;
    float acc = pair_accumulate<KIND>(q, c, d, lane);
    if (lane == 0) out[pair] = pair_finish<KIND>(acc);
  }
}

// backward of pair scoring.  Block per query row: each warp walks candidates j = warp, warp+W, ...
// writing dC[pair,:] and accumulating the row's dQ in registers; warps are then combined in a fixed
// order through shared memory (deterministic, no float atomics).
constexpr int kPairBwdWarps = 8;
template <int KIND>
__global__ void __launch_bounds__(kPairBwdWarps * 32)
pairs_bwd_kernel(const float* __restrict__ Q, const float* __restrict__ table, const void* cand, int idx64,
                 int64_t B, int64_t M, int d, const float* __restrict__ G, const float* __restrict__ scores,
                 float* __restrict__ dQ, float* __restrict__ dC) {
  extern __shared__ float smem[];  // [kPairBwdWarps][d]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int h = d >> 1;
  const int64_t row = blockIdx.x;
  const float* q = Q + row * d;
  float* acc = smem + warp * d;
  for (int k = lane; k < d; k += 32) acc[k] = 0.f;
  __syncwarp();
  for (int64_t j = warp; j < M; j += kPairBwdWarps) {
    const int64_t pair = row * M + j;
    const float g = G[pair];
    const float* c = table + load_index(cand, idx64, pair) * (int64_t)d;
    float* gc = dC + pair * d;
    if (KIND == KGEB_DOT) {
      for (int k = lane; k < d; k += 32) {
        gc[k] = g * q[k];
        acc[k] += g * c[k];
      }
    } else if (KIND == KGEB_NEG_L1) {
      for (int k = lane; k < d; k += 32) {
        float t = -g * sgnf(q[k] - c[k]);
        acc[k] += t;
        gc[k] = -t;
      }
    } else if (KIND == KGEB_NEG_L2 || KIND == KGEB_ROT_L2) {
      const float dist = fabsf(scores[pair]);
      const float coef = dist == 0.f ? 0.f : ((KIND == KGEB_NEG_L2 ? -g : g) / dist);
      for (int k = lane; k < d; k += 32) {
        float t = coef * (q[k] - c[k]);
        acc[k] += t;
        gc[k] = -t;
      }
    } else {  // ROT_L1
      for (int k = lane; k < h; k += 32) {
        float re = q[k] - c[k], im = q[k + h] - c[k + h];
        float m = sqrtf(re * re + im * im);
        float inv = m == 0.f ? 0.f : g / m;
        float tr = re * inv, ti = im * inv;
        acc[k] += tr;
        acc[k + h] += ti;
        gc[k] = -tr;
        gc[k + h] = -ti;
      }
    }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < d; k += blockDim.x) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < kPairBwdWarps; ++w) s += smem[w * d + k];
    dQ[row * d + k] = s;
  }
}

// ------------------------------------------------------------------------------------------
// negative-sampling loss on the [B, 1+N] score rows (column 0 = the positive, train.py:860-868):
//   KL : cross entropy with class 0 (loss.py:195-208)   G = softmax - onehot(0)
//   BCE: sum_j softplus(x+off) - (x_0+off)              G = sigmoid(x+off) - [j == 0]
// one warp per row; writes G (scaled by inv_batch) and the row loss (scaled by inv_batch)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
ns_loss_kernel(int loss, const float* __restrict__ scores, int64_t B, int64_t M, float offset, float inv_batch,
               float* __restrict__ G, float* __restrict__ row_loss) {
  const int lane = threadIdx.x & 31;
  const int64_t row = blockIdx.x * (int64_t)kWarpsPerBlock + (threadIdx.x >> 5);
  if (row >= B) return;
  const float* x = scores + row * M;
  float* g = G + row * M;
  if (loss == KGEB_LOSS_KL) {
    float mx = -INFINITY;
    for (int64_t j = lane; j < M; j += 32) mx = fmaxf(mx, x[j]);
    mx = warp_max(mx);
    float sum = 0.f;
    for (int64_t j = lane; j < M; j += 32) sum += __expf(x[j] - mx);
    sum = warp_sum(sum);
    const float lse = mx + __logf(sum), inv = 1.f / sum;
    for (int64_t j = lane; j < M; j += 32) g[j] = inv_batch * (__expf(x[j] - mx) * inv - (j == 0 ? 1.f : 0.f));
    if (lane == 0) row_loss[row] = inv_batch * (lse - x[0]);
  } else {
    float acc = 0.f;
    for (int64_t j = lane; j < M; j += 32) {
      const float z = x[j] + offset;
      acc += softplusf(z) - (j == 0 ? z : 0.f);
      g[j] = inv_batch * (sigmoidf(z) - (j == 0 ? 1.f : 0.f));
    }
    acc = warp_sum(acc);
    if (lane == 0) row_loss[row] = inv_batch * acc;
  }
}

// ------------------------------------------------------------------------------------------
// One slot of a negative-sampling batch in ONE kernel (train.py:860-999, implementation "triple"): block per positive
// triple -- pair scores of its 1 + N candidates (rows gathered from the L2-resident table), the loss of the row and
// dL/dscores in shared memory, dQ (warps combined in fixed order) and the candidate gradient.  Replaces kgeb_pairs_score +
// kgeb_ns_loss + kgeb_pairs_bwd (three launches, the [B, 1+N] score and gradient matrices through global memory, the
// candidate rows gathered twice from L2 -- the second gather here hits L1).
//   dense == NULL : candidate gradient rows are written to dC[pair, :] for the deterministic sorted scatter (as before);
//   dense != NULL : they are ADDED to dense[cand, :] with vector reductions (red.global.add.v2/v4.f32).  No rows are
//                   materialised and no sort runs, but the order of the additions -- hence the last bits of the sum -- is
//                   not reproducible: the opt-in fast path (deterministic=False).
// ------------------------------------------------------------------------------------------
constexpr int kNsFusedWarps = 8;
__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void red_add_v2(float* addr, float a, float b) {
  asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(addr), "f"(a), "f"(b) : "memory");
}

template <int KIND>
__global__ void __launch_bounds__(kNsFusedWarps * 32)
ns_fused_kernel(int loss, const float* __restrict__ Q, const float* __restrict__ table, const int64_t* __restrict__ cand,
                int64_t B, int64_t M, int d, float offset, float inv_batch, float* __restrict__ dQ, float* __restrict__ dC,
                float* __restrict__ dense, float* __restrict__ row_loss) {
  extern __shared__ float smem[];                 // [kNsFusedWarps][d] dQ partials | [M] scores | [M] dL/dscores
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int h = d >> 1;
  const int64_t row = blockIdx.x;
  const float* q = Q + row * d;
  float* acc = smem + warp * d;
  float* sc = smem + kNsFusedWarps * d;
  float* g_s = sc + M;
  for (int k = lane; k < d; k += 32) acc[k] = 0.f;
  // ---- scores: four candidates of a warp in flight (the loop is L2 latency: index -> row -> shuffle reduction) ----
  for (int64_t j0 = warp; j0 < M; j0 += 4 * kNsFusedWarps) {
    int64_t e[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int64_t j = j0 + u * kNsFusedWarps;
      e[u] = cand[row * M + (j < M ? j : j0)];
    }
    float a[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) a[u] = pair_accumulate_nosum<KIND>(q, table + e[u] * (int64_t)d, d, lane);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float t = warp_sum(a[u]);
      const int64_t j = j0 + u * kNsFusedWarps;
      if (lane == 0 && j < M) sc[j] = pair_finish<KIND>(t);
    }
  }
  __syncthreads();
  // ---- loss of the row and dL/dscores (column 0 is the positive, train.py:864-867); warp 0, as ns_loss_kernel ----
  if (warp == 0) {
    if (loss == KGEB_LOSS_KL) {
      float mx = -INFINITY;
      for (int64_t j = lane; j < M; j += 32) mx = fmaxf(mx, sc[j]);
      mx = warp_max(mx);
      float sum = 0.f;
      for (int64_t j = lane; j < M; j += 32) sum += __expf(sc[j] - mx);
      sum = warp_sum(sum);
      const float lse = mx + __logf(sum), inv = 1.f / sum;
      for (int64_t j = lane; j < M; j += 32) g_s[j] = inv_batch * (__expf(sc[j] - mx) * inv - (j == 0 ? 1.f : 0.f));
      if (lane == 0) row_loss[row] = inv_batch * (lse - sc[0]);
    } else {
      float a = 0.f;
      for (int64_t j = lane; j < M; j += 32) {
        const float z = sc[j] + offset;
        a += softplusf(z) - (j == 0 ? z : 0.f);
        g_s[j] = inv_batch * (sigmoidf(z) - (j == 0 ? 1.f : 0.f));
      }
      a = warp_sum(a);
      if (lane == 0) row_loss[row] = inv_batch * a;
    }
  }
  __syncthreads();
  // ---- backward: dQ partial of this warp, candidate gradient of every pair ----
  int64_t e_next = warp < M ? cand[row * M + warp] : 0;
  for (int64_t j = warp; j < M; j += kNsFusedWarps) {
    const int64_t pair = row * M + j;
    const float g = g_s[j];
    const int64_t e = e_next;
    const float* c = table + e * (int64_t)d;
    float* gc = dense ? dense + e * (int64_t)d : dC + pair * d;
    if (j + kNsFusedWarps < M) {          // the next candidate's row on its way to L1 while this one is processed
      e_next = cand[pair + kNsFusedWarps];
      const float* cn = table + e_next * (int64_t)d;
      for (int k = 4 * lane; k < d; k += 128) asm volatile("prefetch.global.L1 [%0];" ::"l"(cn + k));
    }
    if (KIND == KGEB_ROT_L1 || KIND == KGEB_ROT_L2) {
      // two complex dimensions per lane: re = columns [2k, 2k+2), im = columns [h + 2k, h + 2k + 2)   (d % 4 == 0)
      const float coef2 = KIND == KGEB_ROT_L2 ? (fabsf(sc[j]) == 0.f ? 0.f : g / fabsf(sc[j])) : 0.f;
      for (int k = 2 * lane; k < h; k += 64) {
        const float2 qr = *reinterpret_cast<const float2*>(q + k), qi = *reinterpret_cast<const float2*>(q + h + k);
        const float2 cr = __ldg(reinterpret_cast<const float2*>(c + k)), ci = __ldg(reinterpret_cast<const float2*>(c + h + k));
        float tr[2], ti[2];
        const float re[2] = {qr.x - cr.x, qr.y - cr.y}, im[2] = {qi.x - ci.x, qi.y - ci.y};
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          if (KIND == KGEB_ROT_L1) {
            const float m = sqrtf(re[u] * re[u] + im[u] * im[u]);
            const float inv = m == 0.f ? 0.f : g / m;
            tr[u] = re[u] * inv; ti[u] = im[u] * inv;
          } else {
            tr[u] = coef2 * re[u]; ti[u] = coef2 * im[u];
          }
        }
        acc[k] += tr[0]; acc[k + 1] += tr[1]; acc[h + k] += ti[0]; acc[h + k + 1] += ti[1];
        if (dense) {
          red_add_v2(gc + k, -tr[0], -tr[1]);
          red_add_v2(gc + h + k, -ti[0], -ti[1]);
        } else {
          *reinterpret_cast<float2*>(gc + k) = make_float2(-tr[0], -tr[1]);
          *reinterpret_cast<float2*>(gc + h + k) = make_float2(-ti[0], -ti[1]);
        }
      }
    } else {
      const float dist = fabsf(sc[j]);
      const float coef = KIND == KGEB_NEG_L2 ? (dist == 0.f ? 0.f : -g / dist) : 0.f;
      for (int k = 4 * lane; k < d; k += 128) {                                        // d % 4 == 0
        const float4 qv = *reinterpret_cast<const float4*>(q + k);
        const float4 cv = __ldg(reinterpret_cast<const float4*>(c + k));
        float t[4], o[4];
        const float qa[4] = {qv.x, qv.y, qv.z, qv.w}, ca[4] = {cv.x, cv.y, cv.z, cv.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (KIND == KGEB_DOT) { t[u] = g * ca[u]; o[u] = g * qa[u]; }
          else if (KIND == KGEB_NEG_L1) { t[u] = -g * sgnf(qa[u] - ca[u]); o[u] = -t[u]; }
          else { t[u] = coef * (qa[u] - ca[u]); o[u] = -t[u]; }
          acc[k + u] += t[u];
        }
        if (dense) red_add_v4(gc + k, o[0], o[1], o[2], o[3]);
        else *reinterpret_cast<float4*>(gc + k) = make_float4(o[0], o[1], o[2], o[3]);
      }
    }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < d; k += blockDim.x) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < kNsFusedWarps; ++w) s += smem[w * d + k];
    dQ[row * d + k] = s;
  }
}

// cand[i,0] = target[i]; cand[i,1+j] = negatives[i,j]
__global__ void ns_candidates_kernel(const int64_t* __restrict__ target, const int64_t* __restrict__ neg, int64_t B,
                                     int64_t N, int64_t* __restrict__ cand) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t M = N + 1;
  if (t >= B * M) return;
  const int64_t i = t / M, j = t - i * M;
  cand[t] = j == 0 ? target[i] : neg[i * N + (j - 1)];
}

static int grid_for_rows(int64_t n) {
  int64_t b = (n + kWarpsPerBlock - 1) / kWarpsPerBlock;
  int64_t cap = (int64_t)kNumSMs * 16;
  return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

static int check_model(int model, int d, int l_norm) {
  KGEB_REQUIRE(model >= KGEB_DISTMULT && model <= KGEB_ROTATE, "unknown model id %d", model);
  KGEB_REQUIRE(d > 0, "embedding dim must be positive (got %d)", d);
  if (model == KGEB_COMPLEX || model == KGEB_CP || model == KGEB_SIMPLE || model == KGEB_ROTATE)
    KGEB_REQUIRE((d & 1) == 0, "model %d requires embeddings of even dimensionality (got %d)", model, d);
  if (model == KGEB_TRANSE || model == KGEB_ROTATE) {
    if (l_norm != 1 && l_norm != 2) {
      set_error("l_norm=%d: only l_norm 1 and 2 are built", l_norm);
      return KGEB_ERR_UNSUPPORTED;
    }
  }
  return KGEB_OK;
}

}  // namespace kgeb

using namespace kgeb;

#define DISPATCH_MODEL(model, CALL)                         \
  switch (model) {                                          \
    case KGEB_DISTMULT: { constexpr int M_ = KGEB_DISTMULT; CALL; } break; \
    case KGEB_COMPLEX: { constexpr int M_ = KGEB_COMPLEX; CALL; } break;   \
    case KGEB_CP: { constexpr int M_ = KGEB_CP; CALL; } break;             \
    case KGEB_SIMPLE: { constexpr int M_ = KGEB_SIMPLE; CALL; } break;     \
    case KGEB_RESCAL: { constexpr int M_ = KGEB_RESCAL; CALL; } break;     \
    case KGEB_TRANSE: { constexpr int M_ = KGEB_TRANSE; CALL; } break;     \
    default: { constexpr int M_ = KGEB_ROTATE; CALL; } break;              \
  }

#define DISPATCH_KIND(kind, CALL)                                        \
  switch (kind) {                                                        \
    case KGEB_DOT: { constexpr int K_ = KGEB_DOT; CALL; } break;         \
    case KGEB_NEG_L1: { constexpr int K_ = KGEB_NEG_L1; CALL; } break;   \
    case KGEB_NEG_L2: { constexpr int K_ = KGEB_NEG_L2; CALL; } break;   \
    case KGEB_ROT_L1: { constexpr int K_ = KGEB_ROT_L1; CALL; } break;   \
    default: { constexpr int K_ = KGEB_ROT_L2; CALL; } break;            \
  }

extern "C" {

const char* kgeb_last_error(void) { return g_err; }

int kgeb_version(char* buf, int buflen) {
  if (buf && buflen > 0) snprintf(buf, buflen, "kgeb200 0.1 (sm_100a, cuda %d)", CUDART_VERSION);
  return 100;
}

int kgeb_gather_rows(const float* W, int64_t vocab, int dim, const void* idx, int idx64, int64_t n, float* out,
                     void* stream) {
  KGEB_REQUIRE(W && out && dim > 0 && n >= 0 && vocab >= 0, "gather_rows: bad arguments");
  if (n == 0) return KGEB_OK;
  cudaStream_t st = as_stream(stream);
  const int threads = 256;
  bool v4 = (dim % 4 == 0) && ((reinterpret_cast<uintptr_t>(W) | reinterpret_cast<uintptr_t>(out)) % 16 == 0);
  int64_t work = v4 ? n * (dim / 4) : n * dim;
  int64_t blocks = (work + threads - 1) / threads;
  int64_t cap = (int64_t)kNumSMs * 32;
  int grid = (int)(blocks > cap ? cap : blocks);
  if (v4)
    gather_rows_v4<<<grid, threads, 0, st>>>(reinterpret_cast<const float4*>(W), vocab, dim / 4, idx, idx64, n,
                                             reinterpret_cast<float4*>(out));
  else
    gather_rows_v1<<<grid, threads, 0, st>>>(W, vocab, dim, idx, idx64, n, out);
  KGEB_LAUNCH_CHECK("gather_rows");
  return KGEB_OK;
}

int kgeb_gather_rows_shard(const float* W_shard, int64_t e_lo, int64_t e_hi, int dim, const void* idx, int idx64,
                           int64_t n, float* out, int64_t* local_ids, void* stream) {
  KGEB_REQUIRE(W_shard && idx && out && dim > 0 && n >= 0 && e_lo >= 0 && e_hi >= e_lo, "gather_rows_shard: bad arguments");
  if (n == 0) return KGEB_OK;
  const int64_t blocks = (n * dim + 255) / 256, cap = (int64_t)kNumSMs * 32;
  gather_rows_shard_kernel<<<(int)(blocks > cap ? cap : blocks), 256, 0, as_stream(stream)>>>(W_shard, e_lo, e_hi, dim, idx,
                                                                                             idx64, n, out, local_ids);
  KGEB_LAUNCH_CHECK("gather_rows_shard");
  return KGEB_OK;
}

int kgeb_score_spo(int model, int l_norm, const float* s_src, const void* s_idx, const float* p_src,
                   const void* p_idx, const float* o_src, const void* o_idx, int idx64, int64_t n, int d,
                   float* out, void* stream) {
  int rc = check_model(model, d, l_norm);
  if (rc) return rc;
  KGEB_REQUIRE(s_src && p_src && o_src && out && n >= 0, "score_spo: bad arguments");
  if (n == 0) return KGEB_OK;
  cudaStream_t st = as_stream(stream);
  DISPATCH_MODEL(model, (score_spo_kernel<M_><<<grid_for_rows(n), kWarpsPerBlock * 32, 0, st>>>(
                            l_norm, s_src, s_idx, p_src, p_idx, o_src, o_idx, idx64, n, d, out)));
  KGEB_LAUNCH_CHECK("score_spo");
  return KGEB_OK;
}

int kgeb_score_spo_bwd(int model, int l_norm, const float* s_src, const void* s_idx, const float* p_src,
                       const void* p_idx, const float* o_src, const void* o_idx, int idx64, int64_t n, int d,
                       const float* gout, float* ds, float* dp, float* d_o, void* stream) {
  int rc = check_model(model, d, l_norm);
  if (rc) return rc;
  KGEB_REQUIRE(s_src && p_src && o_src && gout && ds && dp && d_o && n >= 0, "score_spo_bwd: bad arguments");
  if (n == 0) return KGEB_OK;
  cudaStream_t st = as_stream(stream);
  DISPATCH_MODEL(model, (score_spo_bwd_kernel<M_><<<grid_for_rows(n), kWarpsPerBlock * 32, 0, st>>>(
                            l_norm, s_src, s_idx, p_src, p_idx, o_src, o_idx, idx64, n, d, gout, ds, dp, d_o)));
  KGEB_LAUNCH_CHECK("score_spo_bwd");
  return KGEB_OK;
}

int kgeb_query_build(int model, int combine, const int32_t* row_combine, const float* a_src, const void* a_idx,
                     const float* p_src, const void* p_idx, int idx64, int64_t n, int d, float* Q, void* stream) {
  int rc = check_model(model, d, 1);
  if (rc) return rc;
  KGEB_REQUIRE(row_combine || combine == KGEB_SP_ || combine == KGEB__PO, "query_build: combine must be sp_ or _po");
  KGEB_REQUIRE(a_src && p_src && Q && n >= 0, "query_build: bad arguments");
  if (n == 0) return KGEB_OK;
  cudaStream_t st = as_stream(stream);
  DISPATCH_MODEL(model, (query_build_kernel<M_><<<grid_for_rows(n), kWarpsPerBlock * 32, 0, st>>>(
                            combine, row_combine, a_src, a_idx, p_src, p_idx, idx64, n, d, Q)));
  KGEB_LAUNCH_CHECK("query_build");
  return KGEB_OK;
}

int kgeb_query_bwd(int model, int combine, const int32_t* row_combine, const float* a_src, const void* a_idx,
                   const float* p_src, const void* p_idx, int idx64, int64_t n, int d, const float* dQ, float* da,
                   float* dp, void* stream) {
  int rc = check_model(model, d, 1);
  if (rc) return rc;
  KGEB_REQUIRE(row_combine || combine == KGEB_SP_ || combine == KGEB__PO, "query_bwd: combine must be sp_ or _po");
  KGEB_REQUIRE(a_src && p_src && dQ && da && dp && n >= 0, "query_bwd: bad arguments");
  if (n == 0) return KGEB_OK;
  cudaStream_t st = as_stream(stream);
  DISPATCH_MODEL(model, (query_bwd_kernel<M_><<<grid_for_rows(n), kWarpsPerBlock * 32, 0, st>>>(
                            combine, row_combine, a_src, a_idx, p_src, p_idx, idx64, n, d, dQ, da, dp)));
  KGEB_LAUNCH_CHECK("query_bwd");
  return KGEB_OK;
}

int kgeb_pairs_score(int kind, const float* Q, const float* table, const void* cand, int idx64, int64_t B,
                     int64_t M, int d, float* out, void* stream) {
  KGEB_REQUIRE(kind >= KGEB_DOT && kind <= KGEB_ROT_L2, "pairs_score: unknown kind %d", kind);
  KGEB_REQUIRE(Q && table && cand && out && B >= 0 && M >= 0 && d > 0, "pairs_score: bad arguments");
  KGEB_REQUIRE(!(kind >= KGEB_ROT_L1) || (d % 2 == 0), "RotatE requires embeddings of even dimensionality");
  if (B * M == 0) return KGEB_OK;
  cudaStream_t st = as_stream(stream);
  DISPATCH_KIND(kind, (pairs_score_kernel<K_><<<grid_for_rows(B * M), kWarpsPerBlock * 32, 0, st>>>(
                          Q, table, cand, idx64, B, M, d, out)));
  KGEB_LAUNCH_CHECK("pairs_score");
  return KGEB_OK;
}

int kgeb_ns_loss(int loss, const float* scores, int64_t B, int64_t M, float offset, float inv_batch, float* G,
                 float* row_loss, void* stream) {
  KGEB_REQUIRE(loss == KGEB_LOSS_KL || loss == KGEB_LOSS_BCE, "ns_loss: unknown loss %d", loss);
  KGEB_REQUIRE(scores && G && row_loss && B >= 0 && M >= 1, "ns_loss: bad arguments");
  if (B == 0) return KGEB_OK;
  ns_loss_kernel<<<(unsigned)((B + kWarpsPerBlock - 1) / kWarpsPerBlock), kWarpsPerBlock * 32, 0, as_stream(stream)>>>(
      loss, scores, B, M, offset, inv_batch, G, row_loss);
  KGEB_LAUNCH_CHECK("ns_loss");
  return KGEB_OK;
}

int kgeb_ns_candidates(const int64_t* target, const int64_t* negatives, int64_t B, int64_t N, int64_t* cand,
                       void* stream) {
  KGEB_REQUIRE(target && cand && (negatives || N == 0) && B >= 0 && N >= 0, "ns_candidates: bad arguments");
  if (B == 0) return KGEB_OK;
  const int64_t total = B * (N + 1);
  ns_candidates_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(target, negatives, B, N, cand);
  KGEB_LAUNCH_CHECK("ns_candidates");
  return KGEB_OK;
}

int kgeb_pairs_bwd(int kind, const float* Q, const float* table, const void* cand, int idx64, int64_t B,
                   int64_t M, int d, const float* G, const float* scores, float* dQ, float* dC, void* stream) {
  KGEB_REQUIRE(kind >= KGEB_DOT && kind <= KGEB_ROT_L2, "pairs_bwd: unknown kind %d", kind);
  KGEB_REQUIRE(Q && table && cand && G && dQ && dC && B >= 0 && M >= 0 && d > 0, "pairs_bwd: bad arguments");
  KGEB_REQUIRE(!(kind == KGEB_NEG_L2 || kind == KGEB_ROT_L2) || scores, "pairs_bwd: L2 kinds need the scores");
  KGEB_REQUIRE(!(kind >= KGEB_ROT_L1) || (d % 2 == 0), "RotatE requires embeddings of even dimensionality");
  if (B == 0) return KGEB_OK;
  cudaStream_t st = as_stream(stream);
  size_t smem = (size_t)kPairBwdWarps * d * sizeof(float);
  KGEB_REQUIRE(smem <= 48 * 1024, "pairs_bwd: dim %d too large", d);
  DISPATCH_KIND(kind, (pairs_bwd_kernel<K_><<<(unsigned)B, kPairBwdWarps * 32, smem, st>>>(
                          Q, table, cand, idx64, B, M, d, G, scores, dQ, dC)));
  KGEB_LAUNCH_CHECK("pairs_bwd");
  return KGEB_OK;
}

int kgeb_ns_fused(int kind, int loss, const float* Q, const float* table, const int64_t* cand, int64_t B, int64_t M, int d,
                  float offset, float inv_batch, float* dQ, float* dC, float* dense, float* row_loss, void* stream) {
  KGEB_REQUIRE(kind >= KGEB_DOT && kind <= KGEB_ROT_L2, "ns_fused: unknown kind %d", kind);
  KGEB_REQUIRE(loss == KGEB_LOSS_KL || loss == KGEB_LOSS_BCE, "ns_fused: unknown loss %d", loss);
  KGEB_REQUIRE(Q && table && cand && dQ && row_loss && (dC || dense) && B >= 0 && M >= 1 && d > 0, "ns_fused: bad arguments");
  KGEB_REQUIRE(d % 4 == 0, "ns_fused: the embedding dim must be a multiple of 4 (got %d)", d);
  if (B == 0) return KGEB_OK;
  const size_t smem = ((size_t)kNsFusedWarps * d + 2 * (size_t)M) * sizeof(float);
  KGEB_REQUIRE(smem <= 48 * 1024, "ns_fused: dim %d x %lld candidates do not fit the shared memory of a block", d, (long long)M);
  cudaStream_t st = as_stream(stream);
  DISPATCH_KIND(kind, (ns_fused_kernel<K_><<<(unsigned)B, kNsFusedWarps * 32, smem, st>>>(
                          loss, Q, table, cand, B, M, d, offset, inv_batch, dQ, dC, dense, row_loss)));
  KGEB_LAUNCH_CHECK("ns_fused");
  return KGEB_OK;
}

}  // extern "C"
