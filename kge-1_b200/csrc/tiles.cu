// CUDA-core (fp32 FFMA) tile kernels for the all-entity forms: materialised sp_/_po scores, the
// fused score+loss forward/backward (scores never materialised), and the fused score-and-count of
// filtered entity ranking.  These are the exact-fp32 path (KGEB_MATH_FP32, 1e-5 bar) and serve every
// pair kind (DOT / TransE / RotatE); the tcgen05 TF32 tiles for KGEB_DOT live in tc_dot.cu.
//
// Tile = 64 query rows x 64 candidates, 256 threads, 4x4 micro-tile per thread, K staged through
// shared memory in chunks of 16 (k-major so the inner loop reads float4).
#include "common.cuh"

namespace kgeb {

constexpr int BM = 64, BN = 64, BK = 16, TT = 256;

int tc_score_all(const float* Q, int64_t B, int d, const float* table, int64_t m, float* out, int64_t ld,
                 int64_t col_off, cudaStream_t st);  // tc_dot.cu
int64_t tc_stats_partial_bytes(int64_t B, int64_t nnz);                       // tc_dot.cu
int64_t tc_bwd_workspace_bytes(int64_t B, int d, int64_t n_ent, int64_t nnz);  // tc_bwd.cu
bool tc_bwd_supported(int math, int d);                                                    // tc_bwd.cu
int tc_fused_fwd(int loss, int math, const float* Q, const void* Qb, int64_t B, int d, const float* table,
                 const void* tableb, int64_t e_lo, int64_t n_ent, const int64_t* lab_off, const int64_t* lab_col,
                 int64_t nnz, float ls_keep, float ls_add, float offset, float* rowstat, void* ws, int64_t ws_bytes,
                 cudaStream_t st);  // tc_dot.cu
int tc_to_bf16(const float* src, void* dst, int64_t n, cudaStream_t st);  // tc_bwd.cu
int tc_wait_tiles(cudaStream_t st);  // tc_bwd.cu
int tc_label_rows(const float* Q, int64_t B, int d, const float* table, int64_t e_lo, int64_t n_ent, const int64_t* lab_off,
                  const int64_t* lab_col, int64_t nnz, const int32_t* lab_perm, const float* tscale, const float* row_scale,
                  float inv_batch, float* dense_out, void* ws, int64_t ws_bytes, cudaStream_t st,
                  const int64_t* out_rows = nullptr, int64_t n_out = 0);  // tc_bwd.cu
int tc_fused_bwd(int loss, const float* Q, const void* Qb, int64_t B, int d, const float* table, const void* tableb,
                 int64_t e_lo, int64_t n_ent, const int64_t* lab_off, const int64_t* lab_col, int64_t nnz,
                 const int32_t* lab_perm, const float* tscale, float ls_add, float offset, const float* lse,
                 float inv_batch, const float* row_scale, float* dQ, float* dTable, float* rowstat_out, int flags,
                 void* ws, int64_t ws_bytes, cudaStream_t st, const TableUpdate* upd = nullptr);  // tc_bwd.cu
int tc_flash_fwd(const float* Q, const void* Qb, int64_t B, int d, const float* table, const void* tableb, int64_t e_lo,
                 int64_t n_ent, const int64_t* lab_off, const int64_t* lab_col, int64_t nnz, float* rowstat, float* o_sum,
                 int* status, void* ws, int64_t ws_bytes, cudaStream_t st);  // tc_bwd.cu
int tc_flash_dq(const float* Q, int64_t B, int d, const float* table, int64_t e_lo, int64_t n_ent, const int64_t* lab_off,
                const int64_t* lab_col, int64_t nnz, const float* tscale, const float* rowstat_local, const float* lse,
                float inv_batch, const float* row_scale, const float* o_sum, float* dQ, void* ws, int64_t ws_bytes,
                cudaStream_t st);  // tc_bwd.cu
int tc_rank_count(const float* Q, int64_t nq, int d, const float* table, int64_t e_lo, int64_t n_ent,
                  const float* true_score, const void* true_ent, int idx64, const int64_t* f_off,
                  const int64_t* f_col, const int64_t* t_off, const int64_t* t_col, int64_t* counts,
                  cudaStream_t st);  // tc_dot.cu

struct __align__(16) TileSmem {
  float q[2][BK][BM + 4];
  float c[2][BK][BN + 4];
};

// Computes acc[4][4] (+= pair accumulation) for rows row0+ty*4.., candidates col0+tx*4.. .
// Rows/candidates beyond the bounds are loaded as zeros (their results are ignored by callers).
template <int KIND>
__device__ __forceinline__ void tile_accumulate(const float* __restrict__ Q, int64_t B, int64_t row0,
                                                const float* __restrict__ table, const void* cand_idx,
                                                int idx64, int64_t m, int64_t col0, int d, TileSmem& sm,
                                                float (&acc)[4][4]) {
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  constexpr bool kRot = (KIND == KGEB_ROT_L1);
  const int h = d >> 1;
  const int klen = kRot ? h : d;
  // loader mapping: thread -> (row lr = tid/4, k-quad kq = tid%4)
  const int lr = tid >> 2, kq = (tid & 3) * 4;
  const int64_t qrow = row0 + lr;
  const int64_t ccol = col0 + lr;
  const float* qptr = (qrow < B) ? Q + qrow * d : nullptr;
  const float* cptr = (ccol < m) ? table + load_index(cand_idx, idx64, ccol) * (int64_t)d : nullptr;
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const bool vec = ((d & 3) == 0) && (!kRot || (h & 3) == 0);  // rows are 16 B aligned (cudaMalloc + d%4==0)
  for (int k0 = 0; k0 < klen; k0 += BK) {
#pragma unroll
    for (int part = 0; part < (kRot ? 2 : 1); ++part) {
      float qv[4] = {0.f, 0.f, 0.f, 0.f}, cv[4] = {0.f, 0.f, 0.f, 0.f};
      const int k = k0 + kq;
      if (vec) {
        if (k < klen) {
          if (qptr) { float4 t = *reinterpret_cast<const float4*>(qptr + k + part * h); qv[0] = t.x; qv[1] = t.y; qv[2] = t.z; qv[3] = t.w; }
          if (cptr) { float4 t = __ldg(reinterpret_cast<const float4*>(cptr + k + part * h)); cv[0] = t.x; cv[1] = t.y; cv[2] = t.z; cv[3] = t.w; }
        }
      } else {
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (k + u < klen) {
            if (qptr) qv[u] = qptr[k + u + part * h];
            if (cptr) cv[u] = __ldg(cptr + k + u + part * h);
          }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        sm.q[part][kq + u][lr] = qv[u];
        sm.c[part][kq + u][lr] = cv[u];
      }
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float4 a4 = *reinterpret_cast<const float4*>(&sm.q[0][kk][ty * 4]);
      float4 b4 = *reinterpret_cast<const float4*>(&sm.c[0][kk][tx * 4]);
      float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
      float ai[4], bi[4];
      if (kRot) {
        float4 c4 = *reinterpret_cast<const float4*>(&sm.q[1][kk][ty * 4]);
        float4 d4 = *reinterpret_cast<const float4*>(&sm.c[1][kk][tx * 4]);
        ai[0] = c4.x; ai[1] = c4.y; ai[2] = c4.z; ai[3] = c4.w;
        bi[0] = d4.x; bi[1] = d4.y; bi[2] = d4.z; bi[3] = d4.w;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (KIND == KGEB_DOT) {
            acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
          } else if (KIND == KGEB_NEG_L1) {
            acc[i][j] += fabsf(a[i] - b[j]);
          } else if (KIND == KGEB_NEG_L2 || KIND == KGEB_ROT_L2) {
            float t = a[i] - b[j];
            acc[i][j] = fmaf(t, t, acc[i][j]);
          } else {
            float re = a[i] - b[j], im = ai[i] - bi[j];
            acc[i][j] += sqrtf(fmaf(re, re, im * im));
          }
        }
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (KIND == KGEB_NEG_L1) acc[i][j] = -acc[i][j];
      if (KIND == KGEB_NEG_L2) acc[i][j] = -sqrtf(acc[i][j]);
      if (KIND == KGEB_ROT_L2) acc[i][j] = sqrtf(acc[i][j]);
    }
}

// ------------------------------------------------------------------------------------------
// materialised scores
// ------------------------------------------------------------------------------------------
template <int KIND>
__global__ void __launch_bounds__(TT)
score_all_kernel(const float* __restrict__ Q, int64_t B, int d, const float* __restrict__ table,
                 const void* cand_idx, int idx64, int64_t m, float* __restrict__ out, int64_t ld, int64_t col_off) {
  __shared__ TileSmem sm;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int64_t ntc = (m + BN - 1) / BN;
  const int64_t ntr = (B + BM - 1) / BM;
  for (int64_t t = blockIdx.x; t < ntc * ntr; t += gridDim.x) {
    const int64_t row0 = (t / ntc) * BM, col0 = (t % ntc) * BN;
    float acc[4][4];
    tile_accumulate<KIND>(Q, B, row0, table, cand_idx, idx64, m, col0, d, sm, acc);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int64_t r = row0 + ty * 4 + i;
      if (r >= B) continue;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        int64_t c = col0 + tx * 4 + j;
        if (c < m) out[r * ld + col_off + c] = acc[i][j];
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// backward of the materialised form (all kinds; deterministic sequential sums).
// dq kernel: block = 8 query rows, thread = embedding column(s); dc kernel: block = 8 candidates.
// ------------------------------------------------------------------------------------------
template <int KIND>
__device__ __forceinline__ void pair_grad(float g, float x, float qk, float ck, float qk2, float ck2,
                                          float& out1, float& out2) {
  // contribution of pair (q,c) with upstream g and forward score x to d/dq_k (out1) and, for the
  // rotate kinds, d/dq_{k+h} (out2).  d/dc is the negative (distance kinds) or g*q (DOT, handled by caller)
  if (KIND == KGEB_NEG_L1) {
    out1 = -g * sgnf(qk - ck);
  } else if (KIND == KGEB_NEG_L2) {
    float dist = -x;
    out1 = dist == 0.f ? 0.f : -g * (qk - ck) / dist;
  } else if (KIND == KGEB_ROT_L2) {
    out1 = x == 0.f ? 0.f : g * (qk - ck) / x;
  } else if (KIND == KGEB_ROT_L1) {
    float re = qk - ck, im = qk2 - ck2;
    float mm = sqrtf(re * re + im * im);
    float inv = mm == 0.f ? 0.f : g / mm;
    out1 = re * inv;
    out2 = im * inv;
  }
}

constexpr int RB = 8;    // rows (or candidates) per block in the simple backward kernels
constexpr int TCH = 32;  // "other side" items staged per barrier
template <int KIND, bool WRT_Q>
__global__ void __launch_bounds__(128)
score_all_bwd_kernel(const float* __restrict__ Q, int64_t B, int d, const float* __restrict__ table,
                     const void* cand_idx, int idx64, int64_t m, const float* __restrict__ G,
                     const float* __restrict__ X, int64_t ld, int64_t col_off, float* __restrict__ dOut) {
  // WRT_Q: block owns query rows [own0, own0+RB), loops over all candidates.  else: owns candidates.
  const int h = d >> 1;
  constexpr bool kRot = (KIND == KGEB_ROT_L1);
  const int klen = kRot ? h : d;
  const int64_t own0 = (int64_t)blockIdx.x * RB;
  const int64_t n_own = WRT_Q ? B : m;
  const int64_t n_other = WRT_Q ? m : B;
  __shared__ float gs[TCH][RB], xs[TCH][RB];
  __shared__ int64_t other_row[TCH];
  for (int kbase = 0; kbase < klen; kbase += blockDim.x) {  // uniform trip count for every thread
    const int k = kbase + threadIdx.x;
    const bool active = k < klen;
    float own1[RB], own2[RB], acc1[RB], acc2[RB];
#pragma unroll
    for (int r = 0; r < RB; ++r) {
      acc1[r] = acc2[r] = 0.f;
      own1[r] = own2[r] = 0.f;
      int64_t o = own0 + r;
      if (active && o < n_own) {
        const float* p = WRT_Q ? Q + o * d : table + load_index(cand_idx, idx64, o) * (int64_t)d;
        own1[r] = p[k];
        if (kRot) own2[r] = p[k + h];
      }
    }
    for (int64_t t0 = 0; t0 < n_other; t0 += TCH) {
      __syncthreads();
      for (int e = threadIdx.x; e < TCH * RB; e += blockDim.x) {
        int tt = e / RB, r = e % RB;
        int64_t o = own0 + r, t = t0 + tt;
        float g = 0.f, x = 0.f;
        if (o < n_own && t < n_other) {
          int64_t row = WRT_Q ? o : t, col = WRT_Q ? t : o;
          g = G[row * ld + col_off + col];
          if (X) x = X[row * ld + col_off + col];
        }
        gs[tt][r] = g;
        xs[tt][r] = x;
      }
      if (threadIdx.x < TCH) {
        int64_t t = t0 + threadIdx.x;
        other_row[threadIdx.x] = (t < n_other) ? (WRT_Q ? load_index(cand_idx, idx64, t) : t) : 0;
      }
      __syncthreads();
      const int tn = (int)min((int64_t)TCH, n_other - t0);
      if (active) {
        for (int tt = 0; tt < tn; ++tt) {
          const float* p = (WRT_Q ? table : Q) + other_row[tt] * (int64_t)d;
          const float v1 = __ldg(p + k);
          const float v2 = kRot ? __ldg(p + k + h) : 0.f;
#pragma unroll
          for (int r = 0; r < RB; ++r) {
            const float g = gs[tt][r];
            if (KIND == KGEB_DOT) {
              acc1[r] = fmaf(g, v1, acc1[r]);
            } else {
              float o1 = 0.f, o2 = 0.f;
              // pair_grad is written w.r.t. q; w.r.t. c the sign flips and (q,c) = (other, own)
              if (WRT_Q) pair_grad<KIND>(g, xs[tt][r], own1[r], v1, own2[r], v2, o1, o2);
              else       pair_grad<KIND>(g, xs[tt][r], v1, own1[r], v2, own2[r], o1, o2);
              acc1[r] += WRT_Q ? o1 : -o1;
              if (kRot) acc2[r] += WRT_Q ? o2 : -o2;
            }
          }
        }
      }
    }
    if (active) {
#pragma unroll
      for (int r = 0; r < RB; ++r) {
        int64_t o = own0 + r;
        if (o < n_own) {
          dOut[o * d + k] = acc1[r];
          if (kRot) dOut[o * d + k + h] = acc2[r];
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// label cursor: labels of a row are ascending entity ids; tiles are visited in ascending order
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ int64_t lower_bound_i64(const int64_t* a, int64_t lo, int64_t hi, int64_t v) {
  while (lo < hi) {
    int64_t mid = (lo + hi) >> 1;
    if (a[mid] < v) lo = mid + 1; else hi = mid;
  }
  return lo;
}

struct LossParams {
  int loss;            // KGEB_LOSS_*
  float ls_keep;       // 1 - label_smoothing
  float ls_add;        // 1/E if label_smoothing > 0 else 0
  float offset;        // BCE offset
  float inv_batch;     // bwd only
};

// ------------------------------------------------------------------------------------------
// fused forward statistics (all kinds): CTA = (row block, entity chunk); partials to workspace
// rowstat layout per row: [0] KL: running max / BCE: sum softplus(x+off)   [1] KL: sum exp(x-max)
//                         [2] sum_j (x+off)                                 [3] sum over label entries (x+off)
// ------------------------------------------------------------------------------------------
template <int KIND>
__global__ void __launch_bounds__(TT)
fused_fwd_kernel(LossParams lp, const float* __restrict__ Q, int64_t B, int d, const float* __restrict__ table,
                 int64_t e_lo, int64_t n_ent, const int64_t* __restrict__ lab_off,
                 const int64_t* __restrict__ lab_col, int64_t tiles_per_chunk, float* __restrict__ partial) {
  __shared__ TileSmem sm;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int64_t row0 = (int64_t)blockIdx.y * BM;
  const int64_t chunk = blockIdx.x;
  const int64_t ntc = (n_ent + BN - 1) / BN;
  const int64_t t_begin = chunk * tiles_per_chunk;
  const int64_t t_end = min(ntc, t_begin + tiles_per_chunk);
  float s0[4], s1[4], s2[4], s3[4];
  int64_t cur[4], cend[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    s0[i] = (lp.loss == KGEB_LOSS_KL) ? -INFINITY : 0.f;
    s1[i] = s2[i] = s3[i] = 0.f;
    int64_t r = row0 + ty * 4 + i;
    cur[i] = cend[i] = 0;
    if (r < B && lab_off) {
      cend[i] = lab_off[r + 1];
      cur[i] = lower_bound_i64(lab_col, lab_off[r], cend[i], e_lo + t_begin * BN);
    }
  }
  for (int64_t t = t_begin; t < t_end; ++t) {
    const int64_t col0 = t * BN;
    float acc[4][4];
    tile_accumulate<KIND>(Q, B, row0, table, nullptr, 0, n_ent, col0, d, sm, acc);
    const int64_t cbase = col0 + tx * 4;  // first local candidate of this thread
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (lp.loss == KGEB_LOSS_KL) {
        float mx = s0[i];
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (cbase + j < n_ent) mx = fmaxf(mx, acc[i][j]);
        float l = (mx == -INFINITY) ? 0.f : s1[i] * __expf(s0[i] - mx);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (cbase + j < n_ent) {
            l += __expf(acc[i][j] - mx);
            s2[i] += acc[i][j];
          }
        s0[i] = mx;
        s1[i] = l;
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (cbase + j < n_ent) {
            float x = acc[i][j] + lp.offset;
            s0[i] += softplusf(x);
            s2[i] += x;
          }
      }
      // label entries of this row that fall into this tile
      const int64_t tile_hi = e_lo + min(col0 + BN, n_ent);
      while (cur[i] < cend[i]) {
        int64_t c = lab_col[cur[i]];
        if (c >= tile_hi) break;
        int64_t loc = c - e_lo - cbase;
        if (loc >= 0 && loc < 4) {
          float x = (loc == 0 ? acc[i][0] : loc == 1 ? acc[i][1] : loc == 2 ? acc[i][2] : acc[i][3]);
          s3[i] += x + (lp.loss == KGEB_LOSS_BCE ? lp.offset : 0.f);
        }
        ++cur[i];
      }
    }
  }
  // combine the 16 threads (tx) that share rows: lanes differ in the low 4 bits
#pragma unroll
  for (int i = 0; i < 4; ++i) {
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
      float m2 = __shfl_xor_sync(0xffffffffu, s0[i], o);
      float l2 = __shfl_xor_sync(0xffffffffu, s1[i], o);
      if (lp.loss == KGEB_LOSS_KL) {
        float mx = fmaxf(s0[i], m2);
        float a = (s0[i] == -INFINITY) ? 0.f : s1[i] * __expf(s0[i] - mx);
        float b = (m2 == -INFINITY) ? 0.f : l2 * __expf(m2 - mx);
        s0[i] = mx;
        s1[i] = a + b;
      } else {
        s0[i] += m2;
      }
      s2[i] += __shfl_xor_sync(0xffffffffu, s2[i], o);
      s3[i] += __shfl_xor_sync(0xffffffffu, s3[i], o);
    }
    int64_t r = row0 + ty * 4 + i;
    if (tx == 0 && r < B) {
      float* p = partial + (chunk * B + r) * 4;
      p[0] = s0[i]; p[1] = s1[i]; p[2] = s2[i]; p[3] = s3[i];
    }
  }
}

__global__ void fused_fwd_finalize(int loss, const float* __restrict__ partial, int64_t B, int64_t chunks,
                                   float* __restrict__ rowstat) {
  int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (r >= B) return;
  float s0 = (loss == KGEB_LOSS_KL) ? -INFINITY : 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  for (int64_t c = 0; c < chunks; ++c) {  // fixed order -> deterministic
    const float* p = partial + (c * B + r) * 4;
    if (loss == KGEB_LOSS_KL) {
      float mx = fmaxf(s0, p[0]);
      float a = (s0 == -INFINITY) ? 0.f : s1 * __expf(s0 - mx);
      float b = (p[0] == -INFINITY) ? 0.f : p[1] * __expf(p[0] - mx);
      s0 = mx;
      s1 = a + b;
    } else {
      s0 += p[0];
    }
    s2 += p[2];
    s3 += p[3];
  }
  float* o = rowstat + r * 4;
  o[0] = s0; o[1] = s1; o[2] = s2; o[3] = s3;
}

// ------------------------------------------------------------------------------------------
// fused backward (all kinds).  G tile is recomputed in registers, staged in shared memory, and consumed by
// a second phase.  MODE 0: dQ for a (row block, entity chunk) -> partial workspace.
//                  MODE 1: dTable for an entity tile over all row blocks (+= in place).
// The second phase is written for the "own" side (MODE 0: the query rows, MODE 1: the entities) against the "other"
// side, with score_all_bwd_kernel's conventions (pair_grad): d/d own = sum over other of G * f(own - other) with
//   DOT    f = other                               (FFMA)
//   NEG_L1 f = -sign(own - other), sign(0) = 0
//   ROT_L1 f = (own - other) / |own - other|_C per column pair (k, k + d/2), 0 at zero modulus
//   L2     f = (own - other) / x, x the score (-dist / +dist), 0 at zero distance.  1/x is folded into G when it is
//          staged (G'), so the phase is DOT's FFMA plus the row sums of G': d/d own = own * sum G' - sum G' other.
// ------------------------------------------------------------------------------------------
template <int NC>
struct BwdSmem {
  TileSmem t;
  float g[BM][BN + 1];
};

__device__ __forceinline__ void grad_tile(const LossParams& lp, const float (&acc)[4][4], float (&g)[4][4],
                                          const float* lse_or_null, const float* row_scale, int64_t row0,
                                          int64_t B, int64_t col0, int64_t n_ent, int ty, int tx) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int64_t r = row0 + ty * 4 + i;
    float lse = 0.f, rs = lp.inv_batch;
    const float tsum = 1.f;  // sum_j t_ij = 1 for KL targets (L1-normalised rows)
    if (r < B) {
      if (lp.loss == KGEB_LOSS_KL) lse = lse_or_null[r];
      if (row_scale) rs *= row_scale[r];  // upstream d(loss)/d(row loss), stays on the device
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int64_t c = col0 + tx * 4 + j;
      float v = 0.f;
      if (r < B && c < n_ent) {
        if (lp.loss == KGEB_LOSS_KL) v = __expf(acc[i][j] - lse) * tsum - lp.ls_add * tsum;  // dense part of t
        else v = sigmoidf(acc[i][j] + lp.offset) - lp.ls_add;
        v *= rs;
      }
      g[i][j] = v;
    }
  }
}

// Column of accumulator slot c of a lane (d when the slot is unused).  Slots are lane + 32 c; for ROT_L1 the first
// NC / 2 slots hold columns k < d/2 and the last NC / 2 the partner columns k + d/2, so a lane owns whole pairs.
template <int KIND, int NC>
__device__ __forceinline__ int slot_col(int lane, int c, int d) {
  if constexpr (KIND == KGEB_ROT_L1) {
    constexpr int H = NC / 2;
    const int h = d >> 1, k = lane + 32 * (c % H);
    return k < h ? k + (c >= H ? h : 0) : d;
  } else {
    return lane + 32 * c;
  }
}

// out[c] += G * f(own - other) of the L1 kinds (see above) for one (own, other) pair
template <int KIND, int NC>
__device__ __forceinline__ void l1_pair_step(float gv, const float (&own)[NC], const float (&other)[NC],
                                             float (&out)[NC]) {
  if constexpr (KIND == KGEB_NEG_L1) {
#pragma unroll
    for (int c = 0; c < NC; ++c) out[c] = fmaf(-gv, sgnf(own[c] - other[c]), out[c]);
  } else {
    constexpr int H = NC / 2;
#pragma unroll
    for (int c = 0; c < H; ++c) {
      const float re = own[c] - other[c], im = own[c + H] - other[c + H];
      const float m2 = fmaf(re, re, im * im);
      const float inv = m2 == 0.f ? 0.f : gv * rsqrtf(m2);
      out[c] = fmaf(re, inv, out[c]);
      out[c + H] = fmaf(im, inv, out[c + H]);
    }
  }
}

template <int KIND, int NC, int MODE>
__global__ void __launch_bounds__(TT)
fused_bwd_kernel(LossParams lp_in, const float* __restrict__ gscale, const float* __restrict__ Q, int64_t B, int d, const float* __restrict__ table,
                 int64_t e_lo, int64_t n_ent, const int64_t* __restrict__ lab_off,
                 const int64_t* __restrict__ lab_col, const float* __restrict__ lse,
                 const float* __restrict__ tscale, int64_t tiles_per_chunk, float* __restrict__ out) {
  // tscale[r]: weight of one label entry of row r in t (KL: (1-ls)/Z_r ; BCE: (1-ls)); the dense part of
  // t is ls_add (BCE) or ls_add/Z folded by the caller into lp.ls_add == 0 for KL (ls unsupported there).
  constexpr bool kL1 = (KIND == KGEB_NEG_L1 || KIND == KGEB_ROT_L1);
  constexpr bool kL2 = (KIND == KGEB_NEG_L2 || KIND == KGEB_ROT_L2);
  extern __shared__ __align__(16) unsigned char raw[];
  BwdSmem<NC>& sm = *reinterpret_cast<BwdSmem<NC>*>(raw);
  const LossParams lp = lp_in;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int warp = tid >> 5, lane = tid & 31;
  const int64_t ntc = (n_ent + BN - 1) / BN;
  const int64_t ntr = (B + BM - 1) / BM;
  float out_acc[8][NC];
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int c = 0; c < NC; ++c) out_acc[a][c] = 0.f;

  const int64_t outer = MODE == 0 ? (int64_t)blockIdx.y : (int64_t)blockIdx.x;  // row block | entity tile
  // own-side rows of this warp: MODE 0 query rows, MODE 1 entities (local ids)
  const float* own_base = MODE == 0 ? Q : table;
  const int64_t own0 = outer * (MODE == 0 ? BM : BN) + warp * 8, n_own = MODE == 0 ? B : n_ent;
  float own[kL1 ? 8 : 1][kL1 ? NC : 1];   // L1 kinds: own-side operand values, held for the whole block
  float gsum[8];                          // L2 kinds: row sums of G'
#pragma unroll
  for (int a = 0; a < 8; ++a) {
    gsum[a] = 0.f;
    if constexpr (kL1) {
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        const int col = slot_col<KIND, NC>(lane, c, d);
        own[a][c] = (col < d && own0 + a < n_own) ? __ldg(own_base + (own0 + a) * d + col) : 0.f;
      }
    }
  }
  int64_t in_begin, in_end;
  if (MODE == 0) {
    in_begin = (int64_t)blockIdx.x * tiles_per_chunk;
    in_end = min(ntc, in_begin + tiles_per_chunk);
  } else {
    in_begin = 0;
    in_end = ntr;
  }
  for (int64_t inner = in_begin; inner < in_end; ++inner) {
    const int64_t row0 = (MODE == 0 ? outer : inner) * BM;
    const int64_t col0 = (MODE == 0 ? inner : outer) * BN;
    float acc[4][4], g[4][4];
    tile_accumulate<KIND>(Q, B, row0, table, nullptr, 0, n_ent, col0, d, sm.t, acc);
    grad_tile(lp, acc, g, lse, gscale, row0, B, col0, n_ent, ty, tx);
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) sm.g[ty * 4 + i][tx * 4 + j] = g[i][j];
    __syncthreads();
    // subtract the label entries (sparse part of t) that fall into this tile: one thread per row
    if (lab_off && tid < BM) {
      int64_t r = row0 + tid;
      if (r < B) {
        const int64_t hi = lab_off[r + 1];
        const int64_t tile_hi = e_lo + min(col0 + BN, n_ent);
        int64_t p = lower_bound_i64(lab_col, lab_off[r], hi, e_lo + col0);
        const float w = tscale[r] * lp.inv_batch * (gscale ? gscale[r] : 1.f);
        for (; p < hi; ++p) {
          int64_t c = lab_col[p];
          if (c >= tile_hi) break;
          sm.g[tid][c - e_lo - col0] -= w;
        }
      }
    }
    __syncthreads();
    if constexpr (kL2) {
      // G' = G / x with the score x this thread recomputed (zero distance -> zero gradient)
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float& gg = sm.g[ty * 4 + i][tx * 4 + j];
          gg = acc[i][j] == 0.f ? 0.f : gg / acc[i][j];
        }
      __syncthreads();
    }
    if (MODE == 0) {
      // dQ[rows of warp][cols of lane] += sum_j G[row][j] * f(table[col0+j][col])
      const int64_t jn = min((int64_t)BN, n_ent - col0);
      for (int j = 0; j < jn; ++j) {
        const float* crow = table + (col0 + j) * (int64_t)d;
        float cv[NC];
#pragma unroll
        for (int c = 0; c < NC; ++c) {
          int col = slot_col<KIND, NC>(lane, c, d);
          cv[c] = col < d ? __ldg(crow + col) : 0.f;
        }
#pragma unroll
        for (int a = 0; a < 8; ++a) {
          float gv = sm.g[warp * 8 + a][j];
          if constexpr (kL1) {
            l1_pair_step<KIND, NC>(gv, own[a], cv, out_acc[a]);
          } else {
            if constexpr (kL2) gsum[a] += gv;
#pragma unroll
            for (int c = 0; c < NC; ++c) out_acc[a][c] = fmaf(gv, cv[c], out_acc[a][c]);
          }
        }
      }
    } else {
      // dTable[entities of warp][cols of lane] += sum_r G[r][ent] * f(Q[row0+r][col])
      const int64_t rn = min((int64_t)BM, B - row0);
      for (int r = 0; r < rn; ++r) {
        const float* qrow = Q + (row0 + r) * (int64_t)d;
        float qv[NC];
#pragma unroll
        for (int c = 0; c < NC; ++c) {
          int col = slot_col<KIND, NC>(lane, c, d);
          qv[c] = col < d ? __ldg(qrow + col) : 0.f;
        }
#pragma unroll
        for (int a = 0; a < 8; ++a) {
          float gv = sm.g[r][warp * 8 + a];
          if constexpr (kL1) {
            l1_pair_step<KIND, NC>(gv, own[a], qv, out_acc[a]);
          } else {
            if constexpr (kL2) gsum[a] += gv;
#pragma unroll
            for (int c = 0; c < NC; ++c) out_acc[a][c] = fmaf(gv, qv[c], out_acc[a][c]);
          }
        }
      }
    }
    __syncthreads();
  }
  if constexpr (kL2) {   // d/d own = own * sum G' - sum G' other
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        const int col = lane + 32 * c;
        const float ov = (col < d && own0 + a < n_own) ? __ldg(own_base + (own0 + a) * d + col) : 0.f;
        out_acc[a][c] = fmaf(ov, gsum[a], -out_acc[a][c]);
      }
  }
  if (MODE == 0) {
    float* dst = out + ((int64_t)blockIdx.x * B) * d;  // partial [chunk][B][d]
#pragma unroll
    for (int a = 0; a < 8; ++a) {
      int64_t r = outer * BM + warp * 8 + a;
      if (r >= B) continue;
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        int col = slot_col<KIND, NC>(lane, c, d);
        if (col < d) dst[r * d + col] = out_acc[a][c];
      }
    }
  } else {
#pragma unroll
    for (int a = 0; a < 8; ++a) {
      int64_t e = outer * BN + warp * 8 + a;
      if (e >= n_ent) continue;
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        int col = slot_col<KIND, NC>(lane, c, d);
        if (col < d) out[e * d + col] += out_acc[a][c];
      }
    }
  }
}

__global__ void reduce_partials_kernel(const float* __restrict__ partial, int64_t chunks, int64_t numel,
                                       float* __restrict__ out) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  for (; i < numel; i += (int64_t)gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int64_t c = 0; c < chunks; ++c) s += partial[c * numel + i];
    out[i] = s;
  }
}

// ------------------------------------------------------------------------------------------
// fused score-and-count for filtered ranking (all kinds)
// ------------------------------------------------------------------------------------------
template <int KIND>
__global__ void __launch_bounds__(TT)
rank_count_kernel(const float* __restrict__ Q, int64_t nq, int d, const float* __restrict__ table, int64_t e_lo,
                  int64_t n_ent, const float* __restrict__ true_score, const void* true_ent, int idx64,
                  const int64_t* __restrict__ f_off, const int64_t* __restrict__ f_col,
                  const int64_t* __restrict__ t_off, const int64_t* __restrict__ t_col, int64_t tiles_per_chunk,
                  unsigned long long* __restrict__ counts) {
  __shared__ TileSmem sm;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int64_t row0 = (int64_t)blockIdx.y * BM;
  const int64_t ntc = (n_ent + BN - 1) / BN;
  const int64_t t_begin = (int64_t)blockIdx.x * tiles_per_chunk;
  const int64_t t_end = min(ntc, t_begin + tiles_per_chunk);
  int cnt[4][6];
  float tsc[4];
  int64_t tent[4], fcur[4], fend[4], tcur[4], tend[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
#pragma unroll
    for (int k = 0; k < 6; ++k) cnt[i][k] = 0;
    int64_t r = row0 + ty * 4 + i;
    tsc[i] = 0.f; tent[i] = -1; fcur[i] = fend[i] = tcur[i] = tend[i] = 0;
    if (r < nq) {
      float t = true_score[r];
      tsc[i] = (t != t) ? -INFINITY : t;
      tent[i] = load_index(true_ent, idx64, r);
      const int64_t first = e_lo + t_begin * BN;
      if (f_off) { fend[i] = f_off[r + 1]; fcur[i] = lower_bound_i64(f_col, f_off[r], fend[i], first); }
      if (t_off) { tend[i] = t_off[r + 1]; tcur[i] = lower_bound_i64(t_col, t_off[r], tend[i], first); }
    }
  }
  for (int64_t t = t_begin; t < t_end; ++t) {
    const int64_t col0 = t * BN;
    float acc[4][4];
    tile_accumulate<KIND>(Q, nq, row0, table, nullptr, 0, n_ent, col0, d, sm, acc);
    const int64_t cbase = col0 + tx * 4;
    const int64_t tile_hi = e_lo + min(col0 + BN, n_ent);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float ts = tsc[i];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float x = acc[i][j];
        if (e_lo + cbase + j == tent[i]) x = ts;  // entity_ranking.py:170-177
        if (x != x) x = -INFINITY;
        acc[i][j] = x;
        if (cbase + j < n_ent) {
          cnt[i][0] += (x > ts);
          cnt[i][1] += (x == ts);
        }
      }
      // corrections for filtered candidates: their score becomes -inf (entity_ranking.py:499-502)
#pragma unroll
      for (int which = 0; which < 2; ++which) {
        const int64_t* col = which ? t_col : f_col;
        int64_t& cur = which ? tcur[i] : fcur[i];
        const int64_t end = which ? tend[i] : fend[i];
        int64_t prev = -1;
        while (cur < end) {
          int64_t c = col[cur];
          if (c >= tile_hi) break;
          ++cur;
          if (c == prev || c == tent[i]) { prev = c; continue; }
          prev = c;
          int64_t loc = c - e_lo - cbase;
          if (loc >= 0 && loc < 4) {
            float x = (loc == 0 ? acc[i][0] : loc == 1 ? acc[i][1] : loc == 2 ? acc[i][2] : acc[i][3]);
            cnt[i][2 + 2 * which] -= (x > ts);
            cnt[i][3 + 2 * which] += (ts == -INFINITY) - (x == ts);
          }
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int64_t r = row0 + ty * 4 + i;
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      int v = cnt[i][k];
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      cnt[i][k] = v;
    }
    if (tx == 0 && r < nq) {
      unsigned long long* c = counts + r * 6;
      // filtered counts = raw counts + corrections
      long long raw_r = cnt[i][0], raw_t = cnt[i][1];
      atomicAdd(c + 0, (unsigned long long)raw_r);
      atomicAdd(c + 1, (unsigned long long)raw_t);
      atomicAdd(c + 2, (unsigned long long)(raw_r + cnt[i][2]));
      atomicAdd(c + 3, (unsigned long long)(raw_t + cnt[i][3]));
      atomicAdd(c + 4, (unsigned long long)(raw_r + cnt[i][4]));
      atomicAdd(c + 5, (unsigned long long)(raw_t + cnt[i][5]));
    }
  }
}

static int64_t pick_chunks(int64_t ntc, int64_t ntr) {
  // aim at ~2 waves of CTAs over the 148 SMs
  int64_t want = (2 * kNumSMs + ntr - 1) / ntr;
  if (want < 1) want = 1;
  if (want > ntc) want = ntc;
  return want;
}

}  // namespace kgeb

using namespace kgeb;

#define DISPATCH_KIND(kind, CALL)                                        \
  switch (kind) {                                                        \
    case KGEB_DOT: { constexpr int K_ = KGEB_DOT; CALL; } break;         \
    case KGEB_NEG_L1: { constexpr int K_ = KGEB_NEG_L1; CALL; } break;   \
    case KGEB_NEG_L2: { constexpr int K_ = KGEB_NEG_L2; CALL; } break;   \
    case KGEB_ROT_L1: { constexpr int K_ = KGEB_ROT_L1; CALL; } break;   \
    default: { constexpr int K_ = KGEB_ROT_L2; CALL; } break;            \
  }

extern "C" {

int kgeb_score_all(int kind, int math, const float* Q, int64_t B, int d, const float* table,
                   const void* cand_idx, int idx64, int64_t m, float* out, int64_t ld, int64_t col_off,
                   void* stream) {
  KGEB_REQUIRE(kind >= KGEB_DOT && kind <= KGEB_ROT_L2, "score_all: unknown kind %d", kind);
  KGEB_REQUIRE(Q && table && out && B >= 0 && m >= 0 && d > 0 && ld >= col_off + m, "score_all: bad arguments");
  KGEB_REQUIRE(!(kind >= KGEB_ROT_L1) || (d % 2 == 0), "RotatE requires embeddings of even dimensionality");
  if (B == 0 || m == 0) return KGEB_OK;
  cudaStream_t st = as_stream(stream);
  if (math == KGEB_MATH_TF32) {
    KGEB_REQUIRE(kind == KGEB_DOT, "score_all: TF32 tensor tiles exist for KGEB_DOT only");
    KGEB_REQUIRE(cand_idx == nullptr, "score_all: TF32 tiles read the table in place (no candidate subset)");
    return tc_score_all(Q, B, d, table, m, out, ld, col_off, st);
  }
  int64_t tiles = ((m + BN - 1) / BN) * ((B + BM - 1) / BM);
  int grid = (int)(tiles < (int64_t)kNumSMs * 8 ? tiles : (int64_t)kNumSMs * 8);
  DISPATCH_KIND(kind, (score_all_kernel<K_><<<grid, TT, 0, st>>>(Q, B, d, table, cand_idx, idx64, m, out, ld, col_off)));
  KGEB_LAUNCH_CHECK("score_all");
  return KGEB_OK;
}

int kgeb_score_all_bwd(int kind, const float* Q, int64_t B, int d, const float* table, const void* cand_idx,
                       int idx64, int64_t m, const float* G, const float* X, int64_t ld, int64_t col_off,
                       float* dQ, float* dC, void* stream) {
  KGEB_REQUIRE(kind >= KGEB_DOT && kind <= KGEB_ROT_L2, "score_all_bwd: unknown kind %d", kind);
  KGEB_REQUIRE(Q && table && G && B >= 0 && m >= 0 && d > 0, "score_all_bwd: bad arguments");
  KGEB_REQUIRE(!(kind == KGEB_NEG_L2 || kind == KGEB_ROT_L2) || X, "score_all_bwd: L2 kinds need the scores X");
  if (B == 0 || m == 0) return KGEB_OK;
  cudaStream_t st = as_stream(stream);
  if (dQ) {
    unsigned grid = (unsigned)((B + RB - 1) / RB);
    DISPATCH_KIND(kind, (score_all_bwd_kernel<K_, true><<<grid, 128, 0, st>>>(Q, B, d, table, cand_idx, idx64, m, G,
                                                                               X, ld, col_off, dQ)));
    KGEB_LAUNCH_CHECK("score_all_bwd(dQ)");
  }
  if (dC) {
    unsigned grid = (unsigned)((m + RB - 1) / RB);
    DISPATCH_KIND(kind, (score_all_bwd_kernel<K_, false><<<grid, 128, 0, st>>>(Q, B, d, table, cand_idx, idx64, m,
                                                                                G, X, ld, col_off, dC)));
    KGEB_LAUNCH_CHECK("score_all_bwd(dC)");
  }
  return KGEB_OK;
}


static int64_t fused_ws_cuda_core(int64_t B, int d, int64_t num_shard_entities) {
  int64_t ntc = (num_shard_entities + BN - 1) / BN, ntr = (B + BM - 1) / BM;
  if (ntr < 1) ntr = 1;
  int64_t chunks = pick_chunks(ntc < 1 ? 1 : ntc, ntr);
  int64_t a = chunks * B * 4 * (int64_t)sizeof(float);       // fwd partial stats
  int64_t b = chunks * B * (int64_t)d * (int64_t)sizeof(float);  // bwd dQ partials
  int64_t c = B * (int64_t)sizeof(float);                    // per-row label weights
  return (a > b ? a : b) + c + 512;
}

int64_t kgeb_fused_workspace_bytes(int64_t B, int d, int64_t num_shard_entities, int64_t nnz) {
  int64_t a = fused_ws_cuda_core(B, d, num_shard_entities);
  int64_t b = tc_stats_partial_bytes(B, nnz);
  int64_t c = tc_bwd_workspace_bytes(B, d, num_shard_entities, nnz);
  int64_t m = a > b ? a : b;
  m = m > c ? m : c;
  return m + B * 4 + B * (int64_t)d * 2 + 1024;  // + tail: per-row label weights, bf16 mirror of Q
}

// tail of the workspace: [ ... usable ... | bf16 Q mirror | per-row label weights ]
struct TailWs {
  float* tscale;
  void* qb;
  int64_t usable;
};
static TailWs carve_tail(void* ws, int64_t ws_bytes, int64_t B, int d) {
  char* base = reinterpret_cast<char*>(ws);
  char* ts = reinterpret_cast<char*>(reinterpret_cast<uintptr_t>(base + ws_bytes - B * 4) & ~(uintptr_t)255);
  char* qb = reinterpret_cast<char*>(reinterpret_cast<uintptr_t>(ts - B * (int64_t)d * 2) & ~(uintptr_t)255);
  return TailWs{reinterpret_cast<float*>(ts), qb, (int64_t)(qb - base)};
}


__global__ void label_weight_kernel(int loss, const int64_t* __restrict__ lab_off, int64_t B, float ls_keep,
                                    float* __restrict__ tscale) {
  int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (r >= B) return;
  if (loss == KGEB_LOSS_BCE) { tscale[r] = ls_keep; return; }
  int64_t n = lab_off[r + 1] - lab_off[r];  // KL: t = y / ||y||_1  (loss.py:211-213); one-hot for index labels
  tscale[r] = n > 0 ? 1.f / (float)n : 0.f;
}

}  // extern "C"

// fp32 CUDA-core forward statistics of every kind (kgeb_fused_fwd with KGEB_MATH_FP32, kgeb_fused_fwd_kind); B > 0
template <int KIND>
static int fused_fwd_fp32(const LossParams& lp, const float* Q, int64_t B, int d, const float* table, int64_t e_lo,
                          int64_t n_ent, const int64_t* lab_off, const int64_t* lab_col, float* rowstat, void* workspace,
                          cudaStream_t st) {
  const int64_t ntc = (n_ent + BN - 1) / BN, ntr = (B + BM - 1) / BM;
  const int64_t chunks = pick_chunks(ntc < 1 ? 1 : ntc, ntr);
  const int64_t tpc = ntc == 0 ? 1 : (ntc + chunks - 1) / chunks;
  float* partial = reinterpret_cast<float*>(workspace);
  dim3 grid((unsigned)chunks, (unsigned)ntr);
  fused_fwd_kernel<KIND><<<grid, TT, 0, st>>>(lp, Q, B, d, table, e_lo, n_ent, lab_off, lab_col, tpc, partial);
  KGEB_LAUNCH_CHECK("fused_fwd");
  fused_fwd_finalize<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(lp.loss, partial, B, chunks, rowstat);
  KGEB_LAUNCH_CHECK("fused_fwd_finalize");
  return KGEB_OK;
}

template <int KIND, int NC>
static void launch_fused_bwd(const LossParams& lp, const float* grad_scale, const float* Q, int64_t B, int d,
                             const float* table, int64_t e_lo, int64_t n_ent, const int64_t* lab_off,
                             const int64_t* lab_col, const float* lse, const float* tscale, int64_t chunks, int64_t tpc,
                             float* partial, float* dQ, float* dTable, cudaStream_t st) {
  const int64_t ntc = (n_ent + BN - 1) / BN, ntr = (B + BM - 1) / BM;
  size_t smem = sizeof(BwdSmem<NC>);
  cudaFuncSetAttribute(fused_bwd_kernel<KIND, NC, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  cudaFuncSetAttribute(fused_bwd_kernel<KIND, NC, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (dQ) {
    dim3 g0((unsigned)chunks, (unsigned)ntr);
    fused_bwd_kernel<KIND, NC, 0><<<g0, TT, smem, st>>>(lp, grad_scale, Q, B, d, table, e_lo, n_ent, lab_off, lab_col,
                                                         lse, tscale, tpc, partial);
    reduce_partials_kernel<<<(unsigned)((B * d + 255) / 256), 256, 0, st>>>(partial, chunks, B * (int64_t)d, dQ);
  }
  if (dTable && ntc > 0)
    fused_bwd_kernel<KIND, NC, 1><<<(unsigned)ntc, TT, smem, st>>>(lp, grad_scale, Q, B, d, table, e_lo, n_ent, lab_off,
                                                                    lab_col, lse, tscale, tpc, dTable);
}

// fp32 CUDA-core backward of every kind (kgeb_fused_bwd outside the bf16 tiles, kgeb_fused_bwd_kind); B > 0
template <int KIND>
static int fused_bwd_fp32(const LossParams& lp, const float* Q, int64_t B, int d, const float* table, int64_t e_lo,
                          int64_t n_ent, const int64_t* lab_off, const int64_t* lab_col, const float* lse,
                          const float* grad_scale, float* dQ, float* dTable, int flags, void* workspace, cudaStream_t st) {
  const int64_t ntc = (n_ent + BN - 1) / BN, ntr = (B + BM - 1) / BM;
  const int64_t chunks = pick_chunks(ntc < 1 ? 1 : ntc, ntr);
  const int64_t tpc = ntc == 0 ? 1 : (ntc + chunks - 1) / chunks;
  float* partial = reinterpret_cast<float*>(workspace);
  int64_t part_bytes = chunks * B * (int64_t)d * 4, stat_bytes = chunks * B * 16;
  float* tscale = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) +
                                           (((part_bytes > stat_bytes ? part_bytes : stat_bytes) + 255) / 256) * 256);
  label_weight_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(lp.loss, lab_off, B, lp.ls_keep, tscale);
  KGEB_LAUNCH_CHECK("label_weight");
  if (dTable && (flags & KGEB_BWD_OVERWRITE_TABLE) && n_ent > 0)   // the fp32 tiles add: overwrite = clear first
    cudaMemsetAsync(dTable, 0, (size_t)n_ent * d * 4, st);
  // accumulator slots per lane: ceil(d / 32); ROT_L1 2 * ceil(d / 64), whole column pairs per lane
  const int nc = KIND == KGEB_ROT_L1 ? 2 * ((d / 2 + 31) / 32) : (d + 31) / 32;
#define LAUNCH_BWD(NC)                                                                                                    \
  launch_fused_bwd<KIND, NC>(lp, grad_scale, Q, B, d, table, e_lo, n_ent, lab_off, lab_col, lse, tscale, chunks, tpc, \
                             partial, dQ, dTable, st)
  if constexpr (KIND == KGEB_ROT_L1) {
    if (nc <= 2) LAUNCH_BWD(2); else if (nc <= 4) LAUNCH_BWD(4); else LAUNCH_BWD(8);
  } else {
    if (nc <= 1) LAUNCH_BWD(1); else if (nc <= 2) LAUNCH_BWD(2); else if (nc <= 4) LAUNCH_BWD(4); else LAUNCH_BWD(8);
  }
#undef LAUNCH_BWD
  KGEB_LAUNCH_CHECK("fused_bwd");
  return KGEB_OK;
}

extern "C" {

static int check_fused(int loss, int d, float ls, const void* Q, const void* table, int64_t e_lo, int64_t e_hi) {
  KGEB_REQUIRE(loss == KGEB_LOSS_KL || loss == KGEB_LOSS_BCE, "fused: unknown loss %d", loss);
  KGEB_REQUIRE(Q && table && d > 0 && e_hi >= e_lo && e_lo >= 0, "fused: bad arguments");
  if (d > 256) { set_error("fused: entity dim %d > 256 not built (use the materialised path)", d); return KGEB_ERR_UNSUPPORTED; }
  if (loss == KGEB_LOSS_KL && ls != 0.f) {
    set_error("fused: KL with label smoothing is not built (use the materialised path)");
    return KGEB_ERR_UNSUPPORTED;
  }
  return KGEB_OK;
}

int kgeb_fused_fwd(int loss, int math, const float* Q, int64_t B, int d, const float* table, int64_t e_lo,
                   int64_t e_hi, int64_t num_entities, const int64_t* lab_off, const int64_t* lab_col, int64_t nnz,
                   float label_smoothing, float offset, const void* table_bf16, float* rowstat, void* workspace,
                   int64_t workspace_bytes, void* stream) {
  int rc = check_fused(loss, d, label_smoothing, Q, table, e_lo, e_hi);
  if (rc) return rc;
  KGEB_REQUIRE(rowstat, "fused_fwd: rowstat is NULL");
  const int64_t n_ent = e_hi - e_lo;
  if (B == 0) return KGEB_OK;
  cudaStream_t st = as_stream(stream);
  KGEB_REQUIRE(workspace && workspace_bytes >= kgeb_fused_workspace_bytes(B, d, n_ent, nnz), "fused_fwd: workspace too small");
  LossParams lp{loss, 1.f - label_smoothing, label_smoothing > 0.f ? 1.f / (float)num_entities : 0.f, offset, 1.f};
  if (math == KGEB_MATH_TF32 || math == KGEB_MATH_BF16) {
    TailWs tail = carve_tail(workspace, workspace_bytes, B, d);
    if (math == KGEB_MATH_BF16) {
      KGEB_REQUIRE(table_bf16, "fused_fwd(bf16): the bf16 mirror of the table is required (kgeb_to_bf16)");
      if ((rc = tc_to_bf16(Q, tail.qb, B * (int64_t)d, st))) return rc;
    }
    return tc_fused_fwd(loss, math, Q, tail.qb, B, d, table, table_bf16, e_lo, n_ent, lab_off, lab_col, nnz, lp.ls_keep,
                        lp.ls_add, offset, rowstat, workspace, tail.usable, st);
  }
  return fused_fwd_fp32<KGEB_DOT>(lp, Q, B, d, table, e_lo, n_ent, lab_off, lab_col, rowstat, workspace, st);
}

int kgeb_fused_bwd_wait_tiles(void* stream) { return tc_wait_tiles(as_stream(stream)); }

int kgeb_fused_label_rows(int loss, const float* Q, int64_t B, int d, const float* table, int64_t e_lo, int64_t e_hi,
                          const int64_t* lab_off, const int64_t* lab_col, int64_t nnz, const int32_t* lab_perm,
                          float label_smoothing, float inv_batch, const float* grad_scale, float* dTable_out,
                          void* workspace, int64_t workspace_bytes, void* stream) {
  int rc = check_fused(loss, d, label_smoothing, Q, table, e_lo, e_hi);
  if (rc) return rc;
  KGEB_REQUIRE(lab_off && lab_col && dTable_out && workspace, "fused_label_rows: bad arguments");
  KGEB_REQUIRE(d % 4 == 0, "fused_label_rows: entity dim must be a multiple of 4 (got %d)", d);
  if (B == 0 || nnz == 0) return KGEB_OK;
  cudaStream_t st = as_stream(stream);
  const int64_t head = ((B * 4 + 255) / 256) * 256;
  KGEB_REQUIRE(workspace_bytes > head, "fused_label_rows: workspace too small");
  float* tscale = reinterpret_cast<float*>(workspace);
  label_weight_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(loss, lab_off, B, 1.f - label_smoothing, tscale);
  KGEB_LAUNCH_CHECK("label_weight");
  return tc_label_rows(Q, B, d, table, e_lo, e_hi - e_lo, lab_off, lab_col, nnz, lab_perm, tscale, grad_scale, inv_batch,
                       dTable_out, reinterpret_cast<char*>(workspace) + head, workspace_bytes - head, st);
}

// kgeb_fused_label_rows with the rows routed to dense_out[out_rows[i]] ([n_out, d]): the sparse half of the fused update
int kgeb_fused_label_rows_to(int loss, const float* Q, int64_t B, int d, const float* table, int64_t e_lo, int64_t e_hi,
                             const int64_t* lab_off, const int64_t* lab_col, int64_t nnz, const int32_t* lab_perm,
                             float label_smoothing, float inv_batch, const float* grad_scale, const int64_t* out_rows,
                             int64_t n_out, float* dense_out, void* workspace, int64_t workspace_bytes, void* stream) {
  int rc = check_fused(loss, d, label_smoothing, Q, table, e_lo, e_hi);
  if (rc) return rc;
  KGEB_REQUIRE(lab_off && lab_col && dense_out && workspace && out_rows && n_out > 0, "fused_label_rows_to: bad arguments");
  KGEB_REQUIRE(d % 4 == 0, "fused_label_rows_to: entity dim must be a multiple of 4 (got %d)", d);
  if (B == 0 || nnz == 0) return KGEB_OK;
  cudaStream_t st = as_stream(stream);
  const int64_t head = ((B * 4 + 255) / 256) * 256;
  KGEB_REQUIRE(workspace_bytes > head, "fused_label_rows_to: workspace too small");
  float* tscale = reinterpret_cast<float*>(workspace);
  label_weight_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(loss, lab_off, B, 1.f - label_smoothing, tscale);
  KGEB_LAUNCH_CHECK("label_weight");
  return tc_label_rows(Q, B, d, table, e_lo, e_hi - e_lo, lab_off, lab_col, nnz, lab_perm, tscale, grad_scale, inv_batch,
                       dense_out, reinterpret_cast<char*>(workspace) + head, workspace_bytes - head, st, out_rows, n_out);
}

// The dense table gradient of kgeb_fused_bwd (bf16 tiles, no label part) with torch.optim.Adagrad.step applied by the
// tile kernel's flush: rows with slot_of[row] < 0 are updated in place (W, state, bf16 mirror), the others are parked in
// gbuf[slot] for kgeb_touched_update.  Replaces, for an [E, d] table, a stored gradient buffer and an update pass over it
// (2 x E*d*4 bytes of HBM traffic and one launch); reference: train.py:375 optimizer.step() after :323 backward().
}  // extern "C"

// kgeb_fused_bwd_update and its _sched sibling: one tile kernel, clr_dev == NULL selects the by-value rate
static int fused_bwd_update(int loss, const float* Q, int64_t B, int d, float* table, int64_t e_lo, int64_t e_hi,
                            int64_t num_entities, const int64_t* lab_off, float label_smoothing, float offset,
                            const float* lse, float inv_batch, const float* grad_scale, void* table_bf16, float* state,
                            float clr, const float* clr_dev, float eps, const int32_t* slot_of, float* gbuf,
                            const int32_t* skip_flag, void* workspace, int64_t workspace_bytes, void* stream) {
  int rc = check_fused(loss, d, label_smoothing, Q, table, e_lo, e_hi);
  if (rc) return rc;
  KGEB_REQUIRE(tc_bwd_supported(KGEB_MATH_BF16, d), "fused_bwd_update: entity dim must be a multiple of 16 and <= 256 (got %d)", d);
  KGEB_REQUIRE(loss != KGEB_LOSS_KL || lse, "fused_bwd_update: KL needs the per-row log-sum-exp");
  KGEB_REQUIRE(table_bf16 && state && slot_of && gbuf && lab_off, "fused_bwd_update: NULL buffer");
  const int64_t n_ent = e_hi - e_lo;
  if (B == 0 || n_ent == 0) return KGEB_OK;      // zero gradient: Adagrad leaves W and the state as they are
  cudaStream_t st = as_stream(stream);
  KGEB_REQUIRE(workspace && workspace_bytes >= kgeb_fused_workspace_bytes(B, d, n_ent, 0), "fused_bwd_update: workspace too small");
  LossParams lp{loss, 1.f - label_smoothing, label_smoothing > 0.f ? 1.f / (float)num_entities : 0.f, offset, inv_batch};
  TailWs tail = carve_tail(workspace, workspace_bytes, B, d);
  label_weight_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(loss, lab_off, B, lp.ls_keep, tail.tscale);
  KGEB_LAUNCH_CHECK("label_weight");
  if ((rc = tc_to_bf16(Q, tail.qb, B * (int64_t)d, st))) return rc;
  TableUpdate upd{table, state, table_bf16, slot_of, gbuf, skip_flag, clr, eps, clr_dev};
  return tc_fused_bwd(loss, Q, tail.qb, B, d, table, table_bf16, e_lo, n_ent, lab_off, lab_off, 0, nullptr, tail.tscale,
                      lp.ls_add, offset, lse, inv_batch, grad_scale, nullptr, nullptr, nullptr, 0, workspace, tail.usable, st,
                      &upd);
}

extern "C" {

int kgeb_fused_bwd_update(int loss, const float* Q, int64_t B, int d, float* table, int64_t e_lo, int64_t e_hi,
                          int64_t num_entities, const int64_t* lab_off, float label_smoothing, float offset,
                          const float* lse, float inv_batch, const float* grad_scale, void* table_bf16, float* state,
                          float clr, float eps, const int32_t* slot_of, float* gbuf, const int32_t* skip_flag,
                          void* workspace, int64_t workspace_bytes, void* stream) {
  return fused_bwd_update(loss, Q, B, d, table, e_lo, e_hi, num_entities, lab_off, label_smoothing, offset, lse, inv_batch,
                          grad_scale, table_bf16, state, clr, nullptr, eps, slot_of, gbuf, skip_flag, workspace,
                          workspace_bytes, stream);
}

int kgeb_fused_bwd_update_sched(int loss, const float* Q, int64_t B, int d, float* table, int64_t e_lo, int64_t e_hi,
                                int64_t num_entities, const int64_t* lab_off, float label_smoothing, float offset,
                                const float* lse, float inv_batch, const float* grad_scale, void* table_bf16, float* state,
                                const float* clr, float eps, const int32_t* slot_of, float* gbuf, const int32_t* skip_flag,
                                void* workspace, int64_t workspace_bytes, void* stream) {
  KGEB_REQUIRE(clr, "fused_bwd_update_sched: the learning-rate word is NULL");
  return fused_bwd_update(loss, Q, B, d, table, e_lo, e_hi, num_entities, lab_off, label_smoothing, offset, lse, inv_batch,
                          grad_scale, table_bf16, state, 0.f, clr, eps, slot_of, gbuf, skip_flag, workspace, workspace_bytes,
                          stream);
}

int kgeb_fused_bwd(int loss, int math, const float* Q, int64_t B, int d, const float* table, int64_t e_lo,
                   int64_t e_hi, int64_t num_entities, const int64_t* lab_off, const int64_t* lab_col, int64_t nnz,
                   const int32_t* lab_perm, float label_smoothing, float offset, const float* lse, float inv_batch,
                   const float* grad_scale, const void* table_bf16, float* dQ, float* dTable, float* rowstat_out,
                   int flags, void* workspace, int64_t workspace_bytes, void* stream) {
  int rc = check_fused(loss, d, label_smoothing, Q, table, e_lo, e_hi);
  if (rc) return rc;
  KGEB_REQUIRE(loss != KGEB_LOSS_KL || lse, "fused_bwd: KL needs the per-row log-sum-exp");
  KGEB_REQUIRE((flags & ~KGEB_BWD_OVERWRITE_TABLE) == 0, "fused_bwd: unknown flags %d", flags);
  KGEB_REQUIRE(lab_off && lab_col, "fused_bwd: label CSR is NULL");
  const int64_t n_ent = e_hi - e_lo;
  cudaStream_t st = as_stream(stream);
  if (B == 0) {   // no rows: the gradient of an overwritten table is all zeros
    if (dTable && (flags & KGEB_BWD_OVERWRITE_TABLE) && n_ent > 0) cudaMemsetAsync(dTable, 0, (size_t)n_ent * d * 4, st);
    return KGEB_OK;
  }
  KGEB_REQUIRE(workspace && workspace_bytes >= kgeb_fused_workspace_bytes(B, d, n_ent, nnz), "fused_bwd: workspace too small");
  LossParams lp{loss, 1.f - label_smoothing, label_smoothing > 0.f ? 1.f / (float)num_entities : 0.f, offset,
                inv_batch};
  if (tc_bwd_supported(math, d)) {
    KGEB_REQUIRE(table_bf16, "fused_bwd(bf16): the bf16 mirror of the table is required (kgeb_to_bf16)");
    TailWs tail = carve_tail(workspace, workspace_bytes, B, d);
    label_weight_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(loss, lab_off, B, lp.ls_keep, tail.tscale);
    KGEB_LAUNCH_CHECK("label_weight");
    if ((rc = tc_to_bf16(Q, tail.qb, B * (int64_t)d, st))) return rc;
    const bool fused_stats = rowstat_out && dQ && loss == KGEB_LOSS_BCE && n_ent > 0;
    if (rowstat_out && !fused_stats &&
        (rc = kgeb_fused_fwd(loss, math, Q, B, d, table, e_lo, e_hi, num_entities, lab_off, lab_col, nnz, label_smoothing,
                             offset, table_bf16, rowstat_out, workspace, workspace_bytes, stream)))
      return rc;
    return tc_fused_bwd(loss, Q, tail.qb, B, d, table, table_bf16, e_lo, n_ent, lab_off, lab_col, nnz, lab_perm, tail.tscale,
                        lp.ls_add, offset, lse, inv_batch, grad_scale, dQ, dTable, fused_stats ? rowstat_out : nullptr,
                        flags, workspace, tail.usable, st);
  }
  if (rowstat_out && (rc = kgeb_fused_fwd(loss, math, Q, B, d, table, e_lo, e_hi, num_entities, lab_off, lab_col, nnz,
                                          label_smoothing, offset, table_bf16, rowstat_out, workspace, workspace_bytes,
                                          stream)))
    return rc;
  // KGEB_MATH_TF32 (an MN-major TF32 operand would need a second, differently swizzled copy of every tile) and
  // dims outside the BF16 tile build use the fp32 CUDA-core tiles
  return fused_bwd_fp32<KGEB_DOT>(lp, Q, B, d, table, e_lo, n_ent, lab_off, lab_col, lse, grad_scale, dQ, dTable, flags,
                                  workspace, st);
}


// The distance kinds on the fp32 CUDA-core tiles (kgeb_fused_fwd_kind / kgeb_fused_bwd_kind): scores are distances, not
// a GEMM, so there is no tensor-tile or flash form.  Argument errors first, then check_fused's refusals.
static int check_kind(int kind, int d) {
  KGEB_REQUIRE(kind >= KGEB_DOT && kind <= KGEB_ROT_L2, "fused: unknown kind %d", kind);
  KGEB_REQUIRE(!(kind >= KGEB_ROT_L1) || (d % 2 == 0), "RotatE requires embeddings of even dimensionality");
  return KGEB_OK;
}

int kgeb_fused_fwd_kind(int kind, int loss, const float* Q, int64_t B, int d, const float* table, int64_t e_lo,
                        int64_t e_hi, int64_t num_entities, const int64_t* lab_off, const int64_t* lab_col, int64_t nnz,
                        float label_smoothing, float offset, float* rowstat, void* workspace, int64_t workspace_bytes,
                        void* stream) {
  if (kind == KGEB_DOT)
    return kgeb_fused_fwd(loss, KGEB_MATH_FP32, Q, B, d, table, e_lo, e_hi, num_entities, lab_off, lab_col, nnz,
                          label_smoothing, offset, nullptr, rowstat, workspace, workspace_bytes, stream);
  int rc = check_kind(kind, d);
  if (rc) return rc;
  if ((rc = check_fused(loss, d, label_smoothing, Q, table, e_lo, e_hi))) return rc;
  KGEB_REQUIRE(rowstat, "fused_fwd_kind: rowstat is NULL");
  const int64_t n_ent = e_hi - e_lo;
  if (B == 0) return KGEB_OK;
  KGEB_REQUIRE(workspace && workspace_bytes >= kgeb_fused_workspace_bytes(B, d, n_ent, nnz),
               "fused_fwd_kind: workspace too small");
  LossParams lp{loss, 1.f - label_smoothing, label_smoothing > 0.f ? 1.f / (float)num_entities : 0.f, offset, 1.f};
  cudaStream_t st = as_stream(stream);
  DISPATCH_KIND(kind, return fused_fwd_fp32<K_>(lp, Q, B, d, table, e_lo, n_ent, lab_off, lab_col, rowstat, workspace, st));
  return KGEB_OK;
}

int kgeb_fused_bwd_kind(int kind, int loss, const float* Q, int64_t B, int d, const float* table, int64_t e_lo,
                        int64_t e_hi, int64_t num_entities, const int64_t* lab_off, const int64_t* lab_col, int64_t nnz,
                        float label_smoothing, float offset, const float* lse, float inv_batch, const float* grad_scale,
                        float* dQ, float* dTable, int flags, void* workspace, int64_t workspace_bytes, void* stream) {
  if (kind == KGEB_DOT)
    return kgeb_fused_bwd(loss, KGEB_MATH_FP32, Q, B, d, table, e_lo, e_hi, num_entities, lab_off, lab_col, nnz, nullptr,
                          label_smoothing, offset, lse, inv_batch, grad_scale, nullptr, dQ, dTable, nullptr, flags,
                          workspace, workspace_bytes, stream);
  int rc = check_kind(kind, d);
  if (rc) return rc;
  if ((rc = check_fused(loss, d, label_smoothing, Q, table, e_lo, e_hi))) return rc;
  KGEB_REQUIRE(loss != KGEB_LOSS_KL || lse, "fused_bwd_kind: KL needs the per-row log-sum-exp");
  KGEB_REQUIRE((flags & ~KGEB_BWD_OVERWRITE_TABLE) == 0, "fused_bwd_kind: unknown flags %d", flags);
  KGEB_REQUIRE(lab_off && lab_col, "fused_bwd_kind: label CSR is NULL");
  const int64_t n_ent = e_hi - e_lo;
  cudaStream_t st = as_stream(stream);
  if (B == 0) {   // no rows: the gradient of an overwritten table is all zeros
    if (dTable && (flags & KGEB_BWD_OVERWRITE_TABLE) && n_ent > 0) cudaMemsetAsync(dTable, 0, (size_t)n_ent * d * 4, st);
    return KGEB_OK;
  }
  KGEB_REQUIRE(workspace && workspace_bytes >= kgeb_fused_workspace_bytes(B, d, n_ent, nnz),
               "fused_bwd_kind: workspace too small");
  LossParams lp{loss, 1.f - label_smoothing, label_smoothing > 0.f ? 1.f / (float)num_entities : 0.f, offset,
                inv_batch};
  DISPATCH_KIND(kind, return fused_bwd_fp32<K_>(lp, Q, B, d, table, e_lo, n_ent, lab_off, lab_col, lse, grad_scale, dQ,
                                                dTable, flags, workspace, st));
  return KGEB_OK;
}

int kgeb_fused_flash_fwd(const float* Q, int64_t B, int d, const float* table, int64_t e_lo, int64_t e_hi,
                         int64_t num_entities, const int64_t* lab_off, const int64_t* lab_col, int64_t nnz,
                         const void* table_bf16, float* rowstat, float* o_sum, int32_t* status, void* workspace,
                         int64_t workspace_bytes, void* stream) {
  int rc = check_fused(KGEB_LOSS_KL, d, 0.f, Q, table, e_lo, e_hi);
  if (rc) return rc;
  KGEB_REQUIRE(lab_off && lab_col && rowstat && o_sum && table_bf16 && status, "fused_flash_fwd: bad arguments");
  KGEB_REQUIRE(tc_bwd_supported(KGEB_MATH_BF16, d), "fused_flash_fwd: needs the bf16 tiles (dim %% 16 == 0, <= 256; got %d)", d);
  (void)num_entities;
  const int64_t n_ent = e_hi - e_lo;
  if (B == 0) return KGEB_OK;
  cudaStream_t st = as_stream(stream);
  KGEB_REQUIRE(workspace && workspace_bytes >= kgeb_fused_workspace_bytes(B, d, n_ent, nnz), "fused_flash_fwd: workspace too small");
  TailWs tail = carve_tail(workspace, workspace_bytes, B, d);
  if ((rc = tc_to_bf16(Q, tail.qb, B * (int64_t)d, st))) return rc;
  return tc_flash_fwd(Q, tail.qb, B, d, table, table_bf16, e_lo, n_ent, lab_off, lab_col, nnz, rowstat, o_sum, status,
                      workspace, tail.usable, st);
}

int kgeb_fused_flash_dq(const float* Q, int64_t B, int d, const float* table, int64_t e_lo, int64_t e_hi,
                        const int64_t* lab_off, const int64_t* lab_col, int64_t nnz, const float* rowstat_local,
                        const float* lse, float inv_batch, const float* grad_scale, const float* o_sum, float* dQ,
                        void* workspace, int64_t workspace_bytes, void* stream) {
  KGEB_REQUIRE(Q && table && lab_off && lab_col && rowstat_local && lse && o_sum && dQ && d > 0 && e_hi >= e_lo,
               "fused_flash_dq: bad arguments");
  const int64_t n_ent = e_hi - e_lo;
  if (B == 0) return KGEB_OK;
  cudaStream_t st = as_stream(stream);
  KGEB_REQUIRE(workspace && workspace_bytes >= kgeb_fused_workspace_bytes(B, d, n_ent, nnz), "fused_flash_dq: workspace too small");
  TailWs tail = carve_tail(workspace, workspace_bytes, B, d);
  label_weight_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(KGEB_LOSS_KL, lab_off, B, 1.f, tail.tscale);
  KGEB_LAUNCH_CHECK("label_weight");
  return tc_flash_dq(Q, B, d, table, e_lo, n_ent, lab_off, lab_col, nnz, tail.tscale, rowstat_local, lse, inv_batch,
                     grad_scale, o_sum, dQ, workspace, tail.usable, st);
}

// Guard of a captured step whose optimistic path can fail (kgeb_fused_flash_fwd's status): when *flag != 0 the gradient
// buffers are cleared, which makes the Adagrad kernels that follow exact no-ops (state += 0, w -= lr * 0 / ...), so the
// tables and the optimizer state are untouched and the host can repeat the step on the robust path.
__global__ void zero_if_kernel(const int32_t* __restrict__ flag, float4* __restrict__ buf, int64_t n4) {
  if (*flag == 0) return;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x)
    buf[i] = make_float4(0.f, 0.f, 0.f, 0.f);
}

int kgeb_zero_if(const int32_t* flag, float* buf, int64_t numel, void* stream) {
  KGEB_REQUIRE(flag && buf && numel >= 0 && numel % 4 == 0 && (reinterpret_cast<uintptr_t>(buf) & 15) == 0,
               "zero_if: bad arguments (16-byte aligned buffer, multiple of 4 elements)");
  if (numel == 0) return KGEB_OK;
  zero_if_kernel<<<kNumSMs * 4, 256, 0, as_stream(stream)>>>(flag, reinterpret_cast<float4*>(buf), numel / 4);
  KGEB_LAUNCH_CHECK("zero_if");
  return KGEB_OK;
}

// per-row loss values, log-sum-exp and the batch loss from the fused forward statistics: one block, fixed order
__global__ void __launch_bounds__(1024)
loss_rows_kernel(int loss, const float* __restrict__ rowstat, const int64_t* __restrict__ lab_off, int64_t B,
                 float ls_keep, float ls_add, float inv_batch, float* __restrict__ rows_out,
                 float* __restrict__ lse_out, float* __restrict__ total) {
  __shared__ float red[1024];
  float acc = 0.f;
  for (int64_t r = threadIdx.x; r < B; r += blockDim.x) {
    const float* s = rowstat + r * 4;
    const float nnz = (float)(lab_off[r + 1] - lab_off[r]);
    float v, lse = 0.f;
    if (loss == KGEB_LOSS_KL) {
      lse = s[0] + logf(s[1]);
      v = nnz > 0.f ? lse - s[3] / nnz - logf(nnz) : 0.f;   // sum_j t (log t - log_softmax_j), t = y / nnz
    } else {
      v = s[0] - ls_keep * s[3] - ls_add * s[2];           // sum_j softplus(x) - t x, t = keep * y + add
    }
    v *= inv_batch;
    if (rows_out) rows_out[r] = v;
    if (lse_out) lse_out[r] = lse;
    acc += v;
  }
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0 && total) total[0] = red[0];
}

int kgeb_loss_from_rowstat(int loss, const float* rowstat, const int64_t* lab_off, int64_t B, float label_smoothing,
                           int64_t num_entities, float inv_batch, float* rows_out, float* lse_out, float* total,
                           void* stream) {
  KGEB_REQUIRE(loss == KGEB_LOSS_KL || loss == KGEB_LOSS_BCE, "loss_from_rowstat: unknown loss %d", loss);
  KGEB_REQUIRE(rowstat && lab_off && B >= 0, "loss_from_rowstat: bad arguments");
  const float add = label_smoothing > 0.f ? 1.f / (float)num_entities : 0.f;
  loss_rows_kernel<<<1, 1024, 0, as_stream(stream)>>>(loss, rowstat, lab_off, B, 1.f - label_smoothing, add, inv_batch,
                                                      rows_out, lse_out, total);
  KGEB_LAUNCH_CHECK("loss_rows");
  return KGEB_OK;
}

// train.py:747 overwrites the reported avg_loss once per query type: what the job logs for a batch is the value of the
// LAST non-empty query type (sp_ = 0, _po = 1).  out[0] = sum of all rows, out[1] = sum of the rows of the highest type
// present; one block, fixed order.  inv_rel_offset = R > 0: a row with relation id p_idx >= R is a _po query of a
// reciprocal relations model, rewritten to an sp_ query on p + R.
__global__ void __launch_bounds__(1024)
loss_report_kernel(const float* __restrict__ rows_loss, const int32_t* __restrict__ row_type,
                   const int64_t* __restrict__ p_idx, int64_t inv_rel_offset, int64_t B, float* __restrict__ out) {
  __shared__ float red[3][1024];
  float all = 0.f, t1 = 0.f, any1 = 0.f;
  for (int64_t r = threadIdx.x; r < B; r += blockDim.x) {
    const float v = rows_loss[r];
    all += v;
    if (row_type[r] != 0 || (inv_rel_offset > 0 && p_idx[r] >= inv_rel_offset)) { t1 += v; any1 = 1.f; }
  }
  red[0][threadIdx.x] = all; red[1][threadIdx.x] = t1; red[2][threadIdx.x] = any1;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      red[0][threadIdx.x] += red[0][threadIdx.x + o];
      red[1][threadIdx.x] += red[1][threadIdx.x + o];
      red[2][threadIdx.x] += red[2][threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    out[0] = red[0][0];
    out[1] = red[2][0] > 0.f ? red[1][0] : red[0][0];
  }
}

int kgeb_loss_report_inv(const float* rows_loss, const int32_t* row_type, const int64_t* p_idx, int64_t inv_rel_offset,
                         int64_t B, float* out, void* stream) {
  KGEB_REQUIRE(rows_loss && row_type && out && B >= 0, "loss_report: bad arguments");
  KGEB_REQUIRE(inv_rel_offset >= 0 && (inv_rel_offset == 0 || p_idx), "loss_report: inverse relation offset without ids");
  loss_report_kernel<<<1, 1024, 0, as_stream(stream)>>>(rows_loss, row_type, p_idx, inv_rel_offset, B, out);
  KGEB_LAUNCH_CHECK("loss_report");
  return KGEB_OK;
}

int kgeb_loss_report(const float* rows_loss, const int32_t* row_type, int64_t B, float* out, void* stream) {
  return kgeb_loss_report_inv(rows_loss, row_type, nullptr, 0, B, out, stream);
}

int kgeb_to_bf16(const float* src, void* dst, int64_t numel, void* stream) {
  KGEB_REQUIRE(src && dst && numel >= 0, "to_bf16: bad arguments");
  return tc_to_bf16(src, dst, numel, as_stream(stream));
}

int kgeb_rank_count(int kind, int math, const float* Q, int64_t nq, int d, const float* table, int64_t e_lo,
                    int64_t e_hi, const float* true_score, const void* true_ent, int idx64,
                    const int64_t* filt_off, const int64_t* filt_col, const int64_t* test_off,
                    const int64_t* test_col, int64_t* counts, void* stream) {
  KGEB_REQUIRE(kind >= KGEB_DOT && kind <= KGEB_ROT_L2, "rank_count: unknown kind %d", kind);
  KGEB_REQUIRE(Q && table && true_score && true_ent && counts && d > 0 && e_hi >= e_lo, "rank_count: bad arguments");
  KGEB_REQUIRE(!(kind >= KGEB_ROT_L1) || (d % 2 == 0), "RotatE requires embeddings of even dimensionality");
  const int64_t n_ent = e_hi - e_lo;
  if (nq == 0 || n_ent == 0) return KGEB_OK;
  cudaStream_t st = as_stream(stream);
  if (math == KGEB_MATH_TF32) {
    KGEB_REQUIRE(kind == KGEB_DOT, "rank_count: TF32 tensor tiles exist for KGEB_DOT only");
    return tc_rank_count(Q, nq, d, table, e_lo, n_ent, true_score, true_ent, idx64, filt_off, filt_col, test_off,
                         test_col, counts, st);
  }
  const int64_t ntc = (n_ent + BN - 1) / BN, ntr = (nq + BM - 1) / BM;
  const int64_t chunks = pick_chunks(ntc, ntr);
  const int64_t tpc = (ntc + chunks - 1) / chunks;
  dim3 grid((unsigned)chunks, (unsigned)ntr);
  DISPATCH_KIND(kind, (rank_count_kernel<K_><<<grid, TT, 0, st>>>(Q, nq, d, table, e_lo, n_ent, true_score, true_ent,
                                                                   idx64, filt_off, filt_col, test_off, test_col, tpc,
                                                                   reinterpret_cast<unsigned long long*>(counts))));
  KGEB_LAUNCH_CHECK("rank_count");
  return KGEB_OK;
}

}  // extern "C"
