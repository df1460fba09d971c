// tcgen05 backward of the fused all-entity loss for the KGEB_DOT scorers (BF16 operand mirrors, fp32 accumulate
// in tensor memory).  The second GEMM consumes the streamed tile MN-major from the same shared-memory bytes the
// first GEMM reads K-major; tcgen05 allows that for 16-bit operands with the plain 128-byte swizzle (for TF32 an
// MN-major operand needs the SWIZZLE_128B_BASE32B layout, i.e. a second copy of the tile), hence BF16 here.
//
//   G = dL/dS (dense part) is recomputed tile by tile and never leaves the SM:
//     MMA1  S[128 x 64]   = RES[128 x d] * STR[64 x d]^T          (both K-major, TMA 128B-swizzled slabs)
//     epi   G = rs_q * (sigmoid(S+off) - ls_add | exp(S - lse_q))  TMEM -> registers -> swizzled smem
//     MMA2  OUT[128 x d] += G[128 x 64] * STR[64 x d]              (A = G K-major, B = the same STR tile MN-major)
//   with OUT accumulating in tensor memory across the streamed tiles of a job.
//   RES_IS_Q = true : RES = one block of 128 query rows (resident), STR = 64-entity tiles of a chunk of the
//                     table -> OUT = dQ block (partial per chunk, reduced in fixed order afterwards)
//   RES_IS_Q = false: RES = one tile of 128 entities (resident), STR = 64-row tiles of Q (all of them)
//                     -> OUT = G^T Q = dense gradient of those 128 table rows, added to dTable in place.
//   The sparse label part of the target (t_ij at known answers) is linear in G and is applied exactly in
//   fp32 by two small kernels (label_dq_kernel, label rows + sorted scatter), so these kernels carry no
//   CSR logic.
// Warp roles: 0 = TMA producer, 1 = MMA issuer, 2 = TMEM allocator, 4-7 = epilogue (one thread per TMEM lane).
#include "tc_common.cuh"
#include <cuda_bf16.h>
#include <cstdlib>

namespace kgeb {
namespace tcb {

using namespace kgeb::tc;

constexpr int RES_ROWS = 128;                    // UMMA M
// Rows of a streamed tile = UMMA N of MMA1 = K of MMA2.  64 is the measured default.  KGEB_STR_ROWS=128 (tuning build,
// NOT yet run on hardware) halves the per-score cost of everything that is paid per tile -- barrier probes, fences,
// TMEM-load latency -- and issues MMA1 with N = 128 (8 KB of shared-memory operands per 262 k MAC instead of 6 KB per
// 131 k); each epilogue warp then walks its 64 columns in two passes of 32 so that the register budget is unchanged.
#ifndef KGEB_STR_ROWS
#define KGEB_STR_ROWS 64
#endif
constexpr int STR_ROWS = KGEB_STR_ROWS;          // UMMA N of MMA1, K of MMA2
static_assert(STR_ROWS == 64 || STR_ROWS == 128, "KGEB_STR_ROWS must be 64 or 128");
[[maybe_unused]] constexpr int PASSES = STR_ROWS / 64;   // epilogue passes of 32 columns per warp and tile
constexpr int RES_SLAB = RES_ROWS * 128;         // 16 KiB: 128 rows x 128 B
constexpr int STR_SLAB = STR_ROWS * 128;         // 8 KiB:  64 rows x 128 B
constexpr int MAX_STR = 8;                       // streamed-tile ring depth
constexpr int EPQ = 4;                            // epilogue warps per TMEM lane quadrant (latency hiding)
constexpr int NUM_EPI_THREADS = 4 * EPQ * 32;     // 512
constexpr int NUM_THREADS = 128 + NUM_EPI_THREADS;  // warps 0-3: TMA / MMA / TMEM alloc / idle; warps 4-19: epilogue
constexpr int NUM_GROUP_THREADS = NUM_EPI_THREADS / 2;  // two epilogue groups ping-pong on alternate streamed tiles
constexpr int COLS_PER_WARP = 32;                       // S-columns per warp, pass and tile
constexpr int SMEM_BUDGET = 227 * 1024;
constexpr int STAGE_BYTES = RES_ROWS * 128;      // flush staging box of one column part (dTable kernel)

// KGEB_TRACE (tuning builds only): block 0 records (warp, event, tile, clock64) of the pipeline's hand-offs into a global
// buffer read back with kgeb_debug_trace(); tools/trace_bwd.py turns it into a per-tile timeline.
#ifdef KGEB_TRACE
// per-warp slots and a register counter: one fire-and-forget store per event (an atomic slot counter costs an L2 round
// trip of ~850 clk per event and swamps the timeline)
__device__ unsigned long long g_trace[32 << 11];
#define KGEB_TR(ev, u)                                                                                          \
  do {                                                                                                          \
    if (blockIdx.x == 0 && tr_n__ < 2048u)                                                                      \
      g_trace[((threadIdx.x >> 5) << 11) + tr_n__++] =                                                          \
          ((unsigned long long)(ev) << 52) | ((unsigned long long)((u) & 0xfff) << 40) |                         \
          ((unsigned long long)clock64() & 0xffffffffffULL);                                                    \
  } while (0)
#define KGEB_TRW(ev, u) do { if ((threadIdx.x & 31) == 0) KGEB_TR(ev, u); } while (0)
#else
#define KGEB_TR(ev, u)
#define KGEB_TRW(ev, u)
#endif

struct Params {
  int64_t n_res;      // rows of the resident operand (B or shard entities)
  int64_t n_str;      // rows of the streamed operand
  int64_t B;
  int d, ks, nstr;    // ks = ceil(d/32); nstr = ring depth
  int64_t n_res_blocks, n_str_tiles, chunks, tiles_per_chunk;
  int loss;
  float offset, ls_add, inv_batch;
  const float* lse;        // [B] (KL)
  const float* row_scale;  // [B] or NULL
  float* out;              // RES_IS_Q: partial [chunks][B][d] ; else dTable [n_res][d] (+=)
  float* stat_partial;     // STATS: [chunks][4 column parts][B][2] = (sum softplus(x+off), sum (x+off)) over valid entities
  int overwrite;           // !RES_IS_Q: the accumulator is STORED into dTable (plain TMA store) instead of added to it
  const float* mref;       // FLASH: [B] reference score per row (natural units); P = exp(x - mref)
  int a_tmem;              // v2: the resident operand is copied to tensor memory once per job (MMA1 with A in TMEM)
  int* status;             // FLASH: set to 1 when a row sum or an accumulator entry is not finite (reference too low)
  const float* colk;       // !RES_IS_Q, KL: [colk_n] exponent offsets (log(rs_q) - lse_q) * log2(e) per streamed (query) row,
  int colk_n;              //   padded with zeros to a multiple of 64; staged in shared memory by the v2 kernel (0 = unused)
  int colk_n_alloc;        //   floats reserved for it in shared memory (colk_n may be reset to 0 for BCE)
  // !RES_IS_Q, v2: Adagrad in the flush (kgeb_fused_bwd_update).  A finished entity tile holds the COMPLETE dense gradient of
  // its 128 rows; rows that also receive sparse gradient rows this step (upd_slot[row] >= 0) are parked in upd_gbuf[slot]
  // for the row kernel that follows, every other row is updated in place: W, state and the bf16 mirror.
  float* upd_w;            // [n_res, d] fp32 master rows (NULL = no fused update)
  float* upd_state;        // [n_res, d] Adagrad sum of squares
  __nv_bfloat16* upd_mirror;   // [n_res, d] = the resident operand of this kernel (each tile is read once, before its flush)
  const int32_t* upd_slot; // [n_res]
  float* upd_gbuf;         // [slots, d]
  const int* upd_skip;     // non-zero word: the step is being abandoned (failed flash pass) -- touch nothing
  float upd_clr, upd_eps;
  const float* upd_clr_dev;  // non-NULL: the rate is this device word, not upd_clr (read once per update warp)
  int stagger_clk;         // fused update: CTA b starts b * stagger_clk clocks late (see the producer warp of the v2 kernel)
  int upd_debug;           // tuning only (KGEB_UPD_DEBUG): 1 = no loads of W / state, 2 = no stores, 4 = no arithmetic, 8 = no prefetch, 16 = no phase 2
};

// Per-row state of an epilogue thread over one job (one resident row = one TMEM lane).
struct EpiRow {
  float my_rs = 0.f, my_lse = 0.f;            // RES_IS_Q: inv_batch * row_scale and the log-sum-exp of this row
  float fl_m2 = 0.f, fl_l[4] = {0.f, 0.f, 0.f, 0.f};   // FLASH: -mref * log2(e); four partial row sums of P
  // STATS: BCE forward statistics of this (row, column part), summed over the job:
  //   sum softplus(z) = ln2 * sum lg2(1 + e^-|z|) + sum max(z, 0)   (no cancellation between the sums)
  float st_lg = 0.f, st_mx = 0.f, st_x = 0.f;
  int n_pad = 0;
};

// S values of 32 consecutive tile columns (first one = streamed row `qbase`) of this thread's resident row -> G (or P).
template <bool RES_IS_Q, int LOSS, bool HAS_RS, bool STATS, bool FLASH>
__device__ __forceinline__ void epi_math(float (&v)[COLS_PER_WARP], const Params& p, EpiRow& row, const int64_t qbase,
                                         const int lane, const float* kc_s = nullptr) {
  constexpr float kLog2e = 1.4426950408889634f;
  const float off2 = -p.offset * kLog2e;   // ex2(fma(x, -log2e, off2)) = exp(-(x + offset))
  // STATS: entity columns beyond the table end were zero-filled, their score is exactly 0: count them here
  // and take their known contribution (softplus(off), off) out once per job instead of masking per element
  if (STATS || FLASH) row.n_pad += COLS_PER_WARP - (int)max((int64_t)0, min((int64_t)COLS_PER_WARP, p.n_str - qbase));
  // Per-column parameters (columns are query rows when RES is the entity tile): lane c of the warp loads
  // those of column c once per tile, the element loop fetches them with one shuffle.  KL folds everything
  // into one exponent offset:  rs * exp(x - lse) = ex2(x * log2e + kc),  kc = (log(rs) - lse) * log2e.
  float col_k = 0.f, col_rs = row.my_rs;
  if (FLASH) {
    col_k = row.fl_m2;
  } else if (!RES_IS_Q && !(LOSS == KGEB_LOSS_KL && kc_s != nullptr)) {
    const int64_t q = min(qbase + lane, p.B - 1);
    col_rs = HAS_RS ? p.inv_batch * __ldg(p.row_scale + q) : p.inv_batch;
    if (LOSS == KGEB_LOSS_KL) col_k = (__logf(col_rs) - __ldg(p.lse + q)) * kLog2e;
  } else if (LOSS == KGEB_LOSS_KL) {
    col_k = (__logf(row.my_rs) - row.my_lse) * kLog2e;   // rows beyond B: log(0) = -inf -> G = 0
  }
  if (LOSS == KGEB_LOSS_KL && !RES_IS_Q && kc_s != nullptr) {
    // per-column exponent offsets from shared memory (broadcast 128-bit loads: 8 per 32 columns instead of 32 shuffles)
#pragma unroll
    for (int c4 = 0; c4 < COLS_PER_WARP; c4 += 4) {
      const float4 k4 = *reinterpret_cast<const float4*>(kc_s + qbase + c4);
      v[c4] = ex2_ftz(fmaf(v[c4], kLog2e, k4.x));
      v[c4 + 1] = ex2_ftz(fmaf(v[c4 + 1], kLog2e, k4.y));
      v[c4 + 2] = ex2_ftz(fmaf(v[c4 + 2], kLog2e, k4.z));
      v[c4 + 3] = ex2_ftz(fmaf(v[c4 + 3], kLog2e, k4.w));
    }
  } else if (LOSS == KGEB_LOSS_KL) {
#pragma unroll
    for (int c = 0; c < COLS_PER_WARP; ++c) {
      const float kc = RES_IS_Q ? col_k : __shfl_sync(0xffffffffu, col_k, c);
      const float a = fmaf(v[c], kLog2e, kc);
      v[c] = ((c & 7) < KGEB_POLY8_KL) ? ex2_poly<3, false>(a) : ex2_ftz(a);
      if (FLASH) row.fl_l[c & 3] += v[c];
    }
  } else {
    // BCE, four columns per iteration.  MUFU diet (the XU pipe has 16 lanes/clk/SM, the FMA pipe 128; the pipeline
    // trace (tools/trace_bwd.py) shows the epilogue warps spending 55-75 % of a tile in this loop with the XU pipe
    // ~80 % busy, i.e. these kernels are bound by MUFU throughput):
    //  * KGEB_RCP_GROUP = 2 | 4: the reciprocals of a group come from ONE rcp of the product of the group (batch
    //    inversion, 1/a0 = a1 / (a0 a1) ...): 1 MUFU + 3 | 9 FMUL instead of 2 | 4 MUFU; relative error ~4 ulp;
    //  * KGEB_LG2_GROUP = 4..32: sum lg2(a_i) = lg2(prod a_i); a_i in [1, 2], so a product of <= 32 factors stays
    //    far inside the fp32 range and costs one FMUL per factor instead of one MUFU.
    constexpr int RG = KGEB_RCP_GROUP, LG = KGEB_LG2_GROUP;
    static_assert(RG == 1 || RG == 2 || RG == 4, "KGEB_RCP_GROUP must be 1, 2 or 4");
    static_assert(LG == 1 || (LG % 4 == 0 && COLS_PER_WARP % LG == 0), "KGEB_LG2_GROUP must be 1 or a multiple of 4");
    float prod = 1.f;
    const float nls = -p.ls_add;
    // exponent clamp of the non-STATS form: the product of a group must stay finite (the sigmoid of z < -20.8
    // (-41.6) then reads 9e-10 (9e-19), far below the bf16 resolution of G next to any other entry)
    const float tmax = RG == 4 ? 30.f : 60.f;
#pragma unroll
    for (int c = 0; c < COLS_PER_WARP; c += 4) {
      float z[4], e[4], a[4], r[4], rs[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        rs[j] = (!RES_IS_Q && HAS_RS) ? __shfl_sync(0xffffffffu, col_rs, c + j) : col_rs;
        float t;
        if (STATS) {
          // sigmoid and softplus from one exponential, cancellation-free:
          //   e = exp(-|z|), a = 1 + e, r = 1/a;  sigma = z >= 0 ? r : e r;  softplus(z) = max(z,0) + log(a)
          z[j] = v[c + j] + p.offset;
          t = fabsf(z[j]) * -kLog2e;
          e[j] = (((c + j) & 7) < KGEB_POLY8_STATS) ? ex2_poly<4, false>(t) : ex2_ftz(t);
        } else {
          // rs * (sigmoid(x + offset) - ls_add) = rs / (1 + exp(-(x + offset))) - rs ls_add
          t = fmaf(v[c + j], -kLog2e, off2);
          if (RG > 1) t = fminf(t, tmax);
          e[j] = (((c + j) & 7) < KGEB_POLY8_BCE) ? ex2_poly<3, true>(t) : ex2_ftz(t);
        }
        a[j] = 1.f + e[j];
      }
      const float p01 = a[0] * a[1], p23 = a[2] * a[3];
      if (RG == 1) {
#pragma unroll
        for (int j = 0; j < 4; ++j) r[j] = rcp_ftz(a[j]);   // e = inf for very negative z -> rcp gives 0
      } else if (RG == 2) {
        const float i01 = rcp_ftz(p01), i23 = rcp_ftz(p23);
        r[0] = i01 * a[1]; r[1] = i01 * a[0]; r[2] = i23 * a[3]; r[3] = i23 * a[2];
      } else {
        const float ri = rcp_ftz(p01 * p23);
        const float i01 = ri * p23, i23 = ri * p01;
        r[0] = i01 * a[1]; r[1] = i01 * a[0]; r[2] = i23 * a[3]; r[3] = i23 * a[2];
      }
      if (STATS) {
        if (LG > 1) {
          prod *= p01 * p23;
          if (((c + 4) % LG) == 0) {
            row.st_lg += lg2_ftz(prod);
            prod = 1.f;
          }
        } else {
          row.st_lg += (lg2_ftz(a[0]) + lg2_ftz(a[1])) + (lg2_ftz(a[2]) + lg2_ftz(a[3]));
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          row.st_mx += fmaxf(z[j], 0.f);
          row.st_x += z[j];
          v[c + j] = fmaf(z[j] >= 0.f ? r[j] : e[j] * r[j], rs[j], nls * rs[j]);
        }
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[c + j] = fmaf(r[j], rs[j], nls * rs[j]);
      }
    }
  }
}

// FLASH (RES_IS_Q, KL): the forward statistics and the softmax part of dQ in one pass.  The epilogue computes
// P = exp(x - mref_row) against a FIXED per-row reference (a sampled row maximum: bf16 operands and fp32 accumulators keep 8
// exponent bits, so no online rescaling of the accumulator is needed), accumulates the row sums of P in registers and
// OUT += P * STR in tensor memory:  lse = mref + log(sum P),  dQ_dense = rs * exp(mref - lse) * OUT.
template <bool RES_IS_Q, bool BF16, int LOSS, bool HAS_RS, bool STATS, bool FLASH = false>
__global__ void __launch_bounds__(NUM_THREADS, 1)
tc_bwd_kernel(const __grid_constant__ CUtensorMap tm_res, const __grid_constant__ CUtensorMap tm_str,
              const __grid_constant__ CUtensorMap tm_out, const Params p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  // the same base as a shared-window offset: derived from the symbol's shared address (a link-time constant), so the
  // MMA issuers' descriptor arithmetic stays on the uniform datapath (the generic pointer goes through S2R)
  const uint32_t smem_s = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#ifdef KGEB_TRACE
  unsigned tr_n__ = 0;
#endif
  const int KS = p.ks, NSTR = p.nstr;
  constexpr int SLAB_K = Elem<BF16>::kSlabK, UMMA_K = Elem<BF16>::kUmmaK;
  constexpr int G_SLABS = STR_ROWS / SLAB_K;            // K-slabs of the G operand (2 for TF32, 1 for BF16)
  constexpr int G_BYTES = G_SLABS * RES_SLAB;
  uint8_t* res_smem = smem;                                         // [KS] slabs of 16 KiB
  uint8_t* g_smem = res_smem + (size_t)KS * RES_SLAB;               // [2] G buffers
  uint8_t* str_smem = g_smem + 2 * G_BYTES;                         // [NSTR][KS] slabs of 8 KiB
  // !RES_IS_Q: one 16 KiB staging box (128 rows x 32 fp32, 128-byte swizzle) per epilogue column part for the
  // TMA reduce-add flush of the accumulator into the dense table gradient
  uint8_t* stage_smem = str_smem + (size_t)NSTR * KS * STR_SLAB;
  uint64_t* bars = reinterpret_cast<uint64_t*>(stage_smem + (RES_IS_Q ? 0 : EPQ * STAGE_BYTES));
  uint64_t* str_full = bars;                    // [MAX_STR]  TMA -> MMA
  uint64_t* str_empty = bars + MAX_STR;         // [MAX_STR]  MMA2 done -> TMA
  uint64_t* res_full = bars + 2 * MAX_STR;      // TMA -> MMA
  uint64_t* res_empty = res_full + 1;           // job's MMAs done -> TMA
  uint64_t* s_full = res_full + 2;              // [2] MMA1 done -> epilogue
  uint64_t* s_empty = res_full + 4;             // [2] epilogue read S -> MMA
  uint64_t* g_full = res_full + 6;              // [2] epilogue wrote G -> MMA
  uint64_t* g_empty = res_full + 8;             // [2] MMA2 read G -> epilogue
  uint64_t* o_full = res_full + 10;             // job accumulator complete -> epilogue
  uint64_t* o_empty = res_full + 11;            // epilogue flushed -> MMA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_full + 12);
  constexpr int TMEM_COLS = 512;
  constexpr uint32_t S_COL = 0;                 // two S buffers of 64 columns: [0,64), [64,128)
  constexpr uint32_t O_COL = 2 * STR_ROWS;      // OUT accumulator: d <= 256 columns behind the two S buffers
#ifdef KGEB_G_TMEM
  constexpr uint32_t G_COL = 448;               // two G buffers of STR_ROWS / 2 columns at [448, 512)
  static_assert(STR_ROWS == 64, "KGEB_G_TMEM: the G buffers fit behind the accumulator for 64-row tiles only");
#endif

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_res);
    tma_prefetch_desc(&tm_str);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < MAX_STR; ++s) {
      mbar_init(&str_full[s], 1);
      mbar_init(&str_empty[s], 1);
    }
    mbar_init(res_full, 1);
    mbar_init(res_empty, 1);
    for (int b = 0; b < 2; ++b) {
      mbar_init(&s_full[b], 1);
      mbar_init(&s_empty[b], NUM_GROUP_THREADS / 32);
      mbar_init(&g_full[b], NUM_GROUP_THREADS / 32);
      mbar_init(&g_empty[b], 1);
    }
    mbar_init(o_full, 1);
    mbar_init(o_empty, NUM_EPI_THREADS / 32);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<TMEM_COLS>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int64_t n_jobs = p.n_res_blocks * p.chunks;

  if (warp == 0) {
    // ================================ TMA producer ================================
    if (elect_one()) {   // (single elected thread, see the MMA issuers below)
      int slot = 0;
      uint32_t phase = 0, rphase = 0;
      for (int64_t job = blockIdx.x; job < n_jobs; job += gridDim.x) {
        const int64_t rb = job % p.n_res_blocks, ch = job / p.n_res_blocks;
        mbar_wait(res_empty, rphase ^ 1);
        mbar_expect_tx(res_full, (uint32_t)(KS * RES_SLAB));
        for (int k = 0; k < KS; ++k)
          tma_load_2d(res_smem + (size_t)k * RES_SLAB, &tm_res, k * SLAB_K, (int32_t)(rb * RES_ROWS), res_full);
        rphase ^= 1;
        const int64_t u0 = ch * p.tiles_per_chunk, u1 = min(p.n_str_tiles, u0 + p.tiles_per_chunk);
        for (int64_t u = u0; u < u1; ++u) {
          mbar_wait(&str_empty[slot], phase ^ 1);
          mbar_expect_tx(&str_full[slot], (uint32_t)(KS * STR_SLAB));
          for (int k = 0; k < KS; ++k)
            tma_load_2d(str_smem + ((size_t)slot * KS + k) * STR_SLAB, &tm_str, k * SLAB_K, (int32_t)(u * STR_ROWS),
                        &str_full[slot]);
          if (++slot == NSTR) { slot = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA1 issuer: S = RES * STR^T ================================
    // One warp per GEMM: a single issuing thread (barrier probes + descriptor arithmetic + 12 tcgen05.mma per tile)
    // was the critical path of the whole kernel; MMA1 and MMA2 only meet through mbarriers, so they are issued by two
    // warps that run ahead of each other independently.
    // The loop runs under ONE elect.sync predicate: the compiler then knows a single thread executes it and keeps the
    // descriptors in uniform registers (UTCHMMA back to back with one UIADD3.64 between them).  Under `if (lane == 0)`
    // -- or with elect.sync around each instruction -- every tcgen05.mma operand is re-broadcast from vector registers
    // (ELECT / 5x R2UR.BROADCAST / BRA.U.ANY waterfall, 18-19 instructions per MMA): ~150 dependent instructions of a
    // single warp per tile, which the ncu source view showed to be the critical path (epilogue warps spent 26 % of their
    // time waiting for S while the issuer never waited; profiles/README.md).
    if (elect_one()) {
      const uint32_t idesc1 = make_idesc(RES_ROWS, STR_ROWS, 0, 0, Elem<BF16>::kFmt);  // (K-major, K-major)
      const uint64_t dbase = make_desc(0, 16, 1024);
      const uint32_t tbase = tmem_base;
      int slot = 0, sbuf = 0;
      uint32_t ph = 0, sph[2] = {0, 0}, rphase = 0;
      const uint32_t res0 = smem_s, str0 = smem_s + (uint32_t)(KS * RES_SLAB + 2 * G_BYTES);
      for (int64_t job = blockIdx.x; job < n_jobs; job += gridDim.x) {
        const int64_t ch = job / p.n_res_blocks;
        const int64_t u0 = ch * p.tiles_per_chunk, u1 = min(p.n_str_tiles, u0 + p.tiles_per_chunk);
        mbar_wait(res_full, rphase);
        rphase ^= 1;
        for (int64_t u = u0; u < u1; ++u) {
          mbar_wait(&str_full[slot], ph);
          KGEB_TR(1, u);
          mbar_wait(&s_empty[sbuf], sph[sbuf] ^ 1);
          KGEB_TR(2, u);
          tc_fence_after();
          const uint32_t acc = tbase + S_COL + (uint32_t)(sbuf * STR_ROWS);
          for (int k = 0; k < KS; ++k) {
            const uint64_t ra = dbase + (uint64_t)((res0 + (uint32_t)k * RES_SLAB) >> 4);
            const uint64_t sa = dbase + (uint64_t)((str0 + (uint32_t)(slot * KS + k) * STR_SLAB) >> 4);
#pragma unroll
            for (int kk = 0; kk < SLAB_K / UMMA_K; ++kk)   // +32 B (= 2 in descriptor units) per K step
              umma<BF16>(acc, ra + 2 * kk, sa + 2 * kk, idesc1, (k | kk) != 0);
          }
          umma_commit(&s_full[sbuf]);
          KGEB_TR(3, u);
          sph[sbuf] ^= 1;
          sbuf ^= 1;
          if (++slot == NSTR) { slot = 0; ph ^= 1; }
        }
        umma_commit(res_empty);   // all MMA1 of the job issued before this commit have read the resident block
      }
    }
  } else if (warp == 3) {
    // ================================ MMA2 issuer: OUT += G * STR ================================
    if (elect_one()) {
      const uint32_t idesc2 = make_idesc(RES_ROWS, p.d, 0, 1, Elem<BF16>::kFmt);       // (K-major, MN-major)
      const uint64_t abase = make_desc(0, 16, 1024);
      const uint64_t bbase = make_desc(0, STR_SLAB, 1024);
      const uint32_t tbase = tmem_base;
      int slot = 0, gbuf = 0;
      uint32_t gph[2] = {0, 0}, ophase = 0;
      const uint32_t g0 = smem_s + (uint32_t)(KS * RES_SLAB), str0 = g0 + (uint32_t)(2 * G_BYTES);
      const uint32_t acc = tbase + O_COL;
      for (int64_t job = blockIdx.x; job < n_jobs; job += gridDim.x) {
        const int64_t ch = job / p.n_res_blocks;
        const int64_t u0 = ch * p.tiles_per_chunk, u1 = min(p.n_str_tiles, u0 + p.tiles_per_chunk);
        mbar_wait(o_empty, ophase ^ 1);  // previous job's accumulator has been flushed
        for (int64_t u = u0; u < u1; ++u) {
          mbar_wait(&g_full[gbuf], gph[gbuf]);
          KGEB_TR(4, u);
          tc_fence_after();
          const uint32_t ga = g0 + (uint32_t)gbuf * G_BYTES;
          const uint32_t sa = str0 + (uint32_t)(slot * KS) * STR_SLAB;
#pragma unroll
          for (int km = 0; km < STR_ROWS / UMMA_K; ++km) {
            // A: G K-major -- UMMA_K columns = 32 B inside the 128 B row of K-slab (km*UMMA_K / SLAB_K).
            // B: the STR tile MN-major -- UMMA_K K-rows of 128 B (8-row groups 1024 B apart = SBO); N chunks of one
            //    128 B row (SLAB_K columns) are one slab apart (LBO = STR_SLAB).
            const int kcol = km * UMMA_K;
            const uint64_t ad = abase + (uint64_t)((ga + (kcol / SLAB_K) * RES_SLAB + (kcol % SLAB_K) * Elem<BF16>::kBytes) >> 4);
            const uint64_t bd = bbase + (uint64_t)((sa + kcol * 128) >> 4);
#ifdef KGEB_G_TMEM
            (void)ad;
            umma_ts_bf16(acc, tbase + G_COL + (uint32_t)(gbuf * (STR_ROWS / 2) + km * (UMMA_K / 2)), bd, idesc2,
                         !(u == u0 && km == 0));
#else
            umma<BF16>(acc, ad, bd, idesc2, !(u == u0 && km == 0));
#endif
          }
          umma_commit(&str_empty[slot]);  // streamed tile free once MMA2 has read it (MMA1 of it finished long ago)
          umma_commit(&g_empty[gbuf]);
          KGEB_TR(5, u);
          gph[gbuf] ^= 1;
          gbuf ^= 1;
          if (++slot == NSTR) slot = 0;
        }
        umma_commit(o_full);      // accumulator complete
        ophase ^= 1;
      }
    }
  } else if (warp >= 4) {
    // ================================ epilogue ================================
    // 16 warps = 2 groups x (4 lane quadrants x 2 column halves).  Group g owns S/G buffer g, i.e. every other
    // streamed tile: while one group waits on its barriers / TMEM loads the other keeps the MUFU and issue slots busy.
    const int ew = warp - 4;
    const int quad = ew & 3;                               // == warp % 4 : TMEM lane quadrant this warp may access
    const int part = ew >> 2;                              // 0..3
    const int group = part >> 1;                           // buffer / tile parity served by this warp
    const int sub = part & 1;                              // which 32 of the 64 S-columns
    const int trow = quad * 32 + lane;                     // resident row (TMEM lane) of this thread
    const uint32_t lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16);
    uint32_t sph = 0, gph = 0, ophase = 0;                 // phases of this group's buffers
    int64_t gunit = 0;                                     // global tile counter (buffers alternate across jobs too)
    for (int64_t job = blockIdx.x; job < n_jobs; job += gridDim.x) {
      const int64_t rb = job % p.n_res_blocks, ch = job / p.n_res_blocks;
      const int64_t u0 = ch * p.tiles_per_chunk, u1 = min(p.n_str_tiles, u0 + p.tiles_per_chunk);
      const int64_t res_row = rb * RES_ROWS + trow;
      EpiRow er;
      if (FLASH) {
        if (res_row < p.B) er.fl_m2 = -p.mref[res_row] * 1.4426950408889634f;
      } else if (RES_IS_Q && res_row < p.B) {
        er.my_rs = p.inv_batch * (HAS_RS ? p.row_scale[res_row] : 1.f);
        if (LOSS == KGEB_LOSS_KL) er.my_lse = p.lse[res_row];
      }
      for (int64_t u = u0; u < u1; ++u, ++gunit) {
        if ((int)(gunit & 1) != group) continue;
        const int bufi = group;
        KGEB_TRW(8, u);
        mbar_wait(&s_full[bufi], sph);
        KGEB_TRW(9, u);
        sph ^= 1;
        tc_fence_after();
        float v[COLS_PER_WARP];
        tmem_ld32(lane_addr + S_COL + (uint32_t)(bufi * STR_ROWS + sub * COLS_PER_WARP), v);
        tc_fence_before();
        mbar_arrive_warp(&s_empty[bufi]);
        KGEB_TRW(10, u);  // S values are in registers: MMA1 of the tile after next may overwrite them
        // Rows / columns beyond the matrices were zero-filled by TMA, so whatever finite G they get multiplies
        // zeros in MMA2; only the parameter loads are clamped.
        epi_math<RES_IS_Q, LOSS, HAS_RS, STATS, FLASH>(v, p, er, u * STR_ROWS + sub * COLS_PER_WARP, lane);
        KGEB_TRW(11, u);
        mbar_wait(&g_empty[bufi], gph ^ 1);  // MMA2 of this buffer's previous tile has finished reading it
        KGEB_TRW(12, u);
        uint8_t* gb = g_smem + (size_t)bufi * G_BYTES;
        if (BF16) {
          // row trow of the single K-slab: this warp's 32 bf16 = chunks 4*sub .. 4*sub+3 (16 B each), 128-byte swizzle
          // (shared-window address + st.shared: through the generic pointer these are ST.E, resolved in the LSU)
          const uint32_t rowa = smem_s + (uint32_t)(KS * RES_SLAB + bufi * G_BYTES + trow * 128);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            uint32_t w[4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
              asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w[j]) : "f"(v[k * 8 + j * 2 + 1]), "f"(v[k * 8 + j * 2]));
            const int ck = sub * 4 + k;
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(rowa + (uint32_t)((ck ^ (trow & 7)) << 4)),
                         "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3])
                         : "memory");
          }
        } else {
          // TF32: 64 fp32 = two K-slabs of 32 columns; this warp's 32 columns are slab `sub`
          uint8_t* rowp = gb + (size_t)sub * RES_SLAB + (size_t)trow * 128;
#pragma unroll
          for (int ck = 0; ck < 8; ++ck)
            *reinterpret_cast<float4*>(rowp + ((ck ^ (trow & 7)) << 4)) =
                make_float4(v[ck * 4], v[ck * 4 + 1], v[ck * 4 + 2], v[ck * 4 + 3]);
        }
        fence_proxy_async();  // generic-proxy stores -> visible to the tensor core (async proxy)
        mbar_arrive_warp(&g_full[bufi]);
        KGEB_TRW(13, u);
        gph ^= 1;
      }
      if (FLASH && res_row < p.B) {
        // row sum of P over this job's (chunk, column part); zero-filled entity columns beyond the table end scored
        // exactly 0, i.e. P = exp(-mref): taken out once per job
        float* sp = p.stat_partial + (((size_t)ch * 4 + part) * p.B + res_row) * 2;
        const float l = ((er.fl_l[0] + er.fl_l[1]) + (er.fl_l[2] + er.fl_l[3])) - (float)er.n_pad * ex2_ftz(er.fl_m2);
        sp[0] = l;
        sp[1] = 0.f;
        // exp(x - mref) left the fp32 / bf16 range (a score > 88 nats above the reference): the caller re-runs the step
        // with the two-pass kernels (online maximum).  Finite sums are exact whatever their magnitude.
        if (!(fabsf(l) <= 3.0e38f)) *p.status = 1;
      }
      if (STATS && res_row < p.B) {
        float* sp = p.stat_partial + (((size_t)ch * 4 + part) * p.B + res_row) * 2;
        const float zp = p.offset;
        const float st_sp = fmaf(0.69314718f, er.st_lg, er.st_mx);
        sp[0] = st_sp - (float)er.n_pad * fmaf(0.69314718f, __log2f(1.f + __expf(-fabsf(zp))), fmaxf(zp, 0.f));
        sp[1] = er.st_x - (float)er.n_pad * zp;
      }
      // flush the job's accumulator
      mbar_wait(o_full, ophase);
      ophase ^= 1;
      tc_fence_after();
      if (RES_IS_Q) {
        // partial dQ of this chunk: plain stores, 16-column groups dealt round-robin to the column parts
        for (int c0 = part * 16; c0 < p.d; c0 += 16 * EPQ) {
          float o[16];
          tmem_ld16(lane_addr + O_COL + (uint32_t)c0, o);
          if (res_row < p.n_res) {
            float* dst = p.out + ((size_t)ch * p.B + res_row) * p.d + c0;
            float big = 0.f;
#pragma unroll
            for (int c = 0; c < 16; c += 4) {
              *reinterpret_cast<float4*>(dst + c) = make_float4(o[c], o[c + 1], o[c + 2], o[c + 3]);
              if (FLASH) big = fmaxf(fmaxf(big, fmaxf(fabsf(o[c]), fabsf(o[c + 1]))), fmaxf(fabsf(o[c + 2]), fabsf(o[c + 3])));
            }
            if (FLASH && !(big <= 3.0e38f)) *p.status = 1;   // inf or NaN in the accumulator
          }
        }
      } else {
        // dense table gradient += accumulator.  A thread-per-row read-modify-write of global memory is uncoalesced
        // and keeps the whole pipeline waiting on HBM round trips once per job; instead each column part stages
        // 32-column boxes in swizzled shared memory and one thread hands them to the TMA as reduce-adds (the add
        // happens in L2, asynchronously; this CTA is the only writer of these rows, so the result is deterministic).
        uint8_t* stage = stage_smem + (size_t)part * STAGE_BYTES;
        const bool leader = (quad == 0 && lane == 0);
        const int nbox = (p.d + 31) / 32;
        for (int box = part; box < nbox; box += EPQ) {
          if (leader) bulk_wait_read0();             // the previous store from this staging box has read it
          named_bar_sync(1 + part, 128);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            float o[16];
            tmem_ld16(lane_addr + O_COL + (uint32_t)(box * 32 + h * 16), o);
            uint8_t* rowp = stage + (size_t)trow * 128;
#pragma unroll
            for (int j = 0; j < 4; ++j)
              *reinterpret_cast<float4*>(rowp + (((h * 4 + j) ^ (trow & 7)) << 4)) =
                  make_float4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
          }
          fence_proxy_async();
          named_bar_sync(1 + part, 128);
          if (leader) {
            // rows / columns past the end are clipped.  overwrite: this CTA is the only writer of these rows and K (all
            // query tiles) is complete, so a plain store does -- no cleared buffer, no read-modify-write in L2
            if (p.overwrite) tma_store_2d(&tm_out, stage, box * 32, (int32_t)(rb * RES_ROWS));
            else tma_reduce_add_2d(&tm_out, stage, box * 32, (int32_t)(rb * RES_ROWS));
            bulk_commit();
          }
        }
      }
      tc_fence_before();
      mbar_arrive_warp(o_empty);
    }
  }

  if (!RES_IS_Q && warp >= 4 && ((warp - 4) & 3) == 0 && lane == 0) bulk_wait0();  // outstanding reduce-adds
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}


// ---------------------------------------------------------------------------------------------
// v2 pipeline (default): FOUR streamed tiles in flight, G handed to MMA2 through tensor memory.
//
// What the pipeline traces of the kernel above showed (profiles/README.md): neither the tensor pipe (~512 clk of MMA per
// 128x64 tile) nor the MUFU pipe (512 clk) is the limit -- a tile takes ~1000 clk because only two tiles are in the
// epilogue at any time and each of them walks a ~1200 clk dependent chain (barrier -> TMEM load -> math -> shared-memory
// store -> proxy fence -> barrier).  Here
//   * tensor memory holds FOUR S buffers of 64 columns + the OUT accumulator (4*64 + d <= 512 columns);
//   * the 16 epilogue warps form four groups of four (one warp per TMEM lane quadrant); group g owns buffer g and every
//     fourth tile, so the four warps of an SM sub-partition are always in four different phases of the chain;
//   * a warp handles all 64 columns of its 32 rows in two passes of 32 (same register footprint as before);
//   * G (bf16) is written back with tcgen05.st INTO THE FIRST 32 COLUMNS OF THE S BUFFER IT CAME FROM (all of S has been
//     read by then) and MMA2 takes it from there as its A operand (tcgen05.mma with A in tensor memory): no shared-memory
//     round trip of G (32 KB of the 112 KB of shared-memory traffic per tile), no generic->async proxy fence, and the
//     "S consumed" / "G consumed" barriers collapse into one (MMA2's commit frees the buffer for MMA1 of tile u + 4);
//   * the shared memory G occupied goes to the streamed-tile ring.
// ---------------------------------------------------------------------------------------------
constexpr int NG = 4;   // tiles in flight = S/G buffers = epilogue groups

// Register split of the 768-thread fused-update kernel.  The pool is what the CTA got at launch (768 x 80 = 61440): the
// epilogue warps can only grow by what the other two warpgroups release, 128 c + 512 e + 128 u <= 61440.  (A first version
// asked for 40 / 96 / 72 = 63488: the fourth epilogue warpgroup waited for registers forever.)
#ifndef KGEB_UPD_REG_CTRL
#define KGEB_UPD_REG_CTRL 40
#define KGEB_UPD_REG_EPI 88
#define KGEB_UPD_REG_UPD 88
#endif
static_assert(128 * KGEB_UPD_REG_CTRL + 512 * KGEB_UPD_REG_EPI + 128 * KGEB_UPD_REG_UPD <= 768 * 80, "register pool of the CTA");
__device__ __forceinline__ float sqrt_approx(float x) { float y; asm("sqrt.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
constexpr int UPD_THREADS = 128;   // fused update: one more warpgroup, warp 20 + p applies Adagrad to the box of column part p

template <int N>
__device__ __forceinline__ void setmaxnreg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }

template <bool RES_IS_Q, int LOSS, bool HAS_RS, bool STATS, bool FLASH = false, bool UPD = false>
__global__ void __launch_bounds__(NUM_THREADS + (UPD ? UPD_THREADS : 0), 1)
tc_bwd4_kernel(const __grid_constant__ CUtensorMap tm_res, const __grid_constant__ CUtensorMap tm_str,
               const __grid_constant__ CUtensorMap tm_out, const Params p) {
  static_assert(STR_ROWS == 64, "the v2 pipeline is laid out for 64-row streamed tiles");
  constexpr bool BF16 = true;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const uint32_t smem_s = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int KS = p.ks, NSTR = p.nstr;
  constexpr int SLAB_K = Elem<BF16>::kSlabK, UMMA_K = Elem<BF16>::kUmmaK;
  uint8_t* res_smem = smem;                                         // [KS] slabs of 16 KiB
  uint8_t* str_smem = res_smem + (size_t)KS * RES_SLAB;             // [NSTR][KS] slabs of 8 KiB
  uint8_t* stage_smem = str_smem + (size_t)NSTR * KS * STR_SLAB;    // !RES_IS_Q: flush staging boxes
  uint64_t* bars = reinterpret_cast<uint64_t*>(stage_smem + (RES_IS_Q ? 0 : EPQ * STAGE_BYTES));
  uint64_t* str_full = bars;                    // [MAX_STR]  TMA -> MMA1
  uint64_t* str_empty = bars + MAX_STR;         // [MAX_STR]  MMA2 done -> TMA
  uint64_t* res_full = bars + 2 * MAX_STR;      // TMA -> MMA1
  uint64_t* res_empty = res_full + 1;           // job's MMA1s done -> TMA
  uint64_t* s_full = res_full + 2;              // [NG] MMA1 done -> epilogue group
  uint64_t* g_full = s_full + NG;               // [NG] epilogue group wrote G -> MMA2
  uint64_t* buf_free = g_full + NG;             // [NG] MMA2 read G -> MMA1 may overwrite the buffer
  uint64_t* o_full = buf_free + NG;             // job accumulator complete -> epilogue
  uint64_t* o_empty = o_full + 1;               // epilogue flushed -> MMA2
  uint64_t* a_full = o_empty + 1;               // a_tmem: epilogue copied the resident block to tensor memory -> MMA1
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_full + 1);
  uint64_t* stage_full = a_full + 2;            // UPD [EPQ]: the part's epilogue warps staged the gradient box -> update warp
  uint64_t* stage_free = stage_full + EPQ;      // UPD [EPQ]: update warp has consumed the staging box (and its slots)
  // !RES_IS_Q, KL: the per-query exponent offsets of ALL streamed rows (the same for every job), 16-byte aligned
  float* kc_smem = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 512);
  const float* kc_s = (!RES_IS_Q && LOSS == KGEB_LOSS_KL && p.colk_n > 0) ? kc_smem : nullptr;
  if (kc_s)
    for (int i = threadIdx.x; i < p.colk_n; i += blockDim.x) kc_smem[i] = p.colk[i];
  int32_t* slot_s = reinterpret_cast<int32_t*>(kc_smem + p.colk_n_alloc);   // !RES_IS_Q: [EPQ][RES_ROWS] (fused update) + rate
  constexpr int TMEM_COLS = 512;
  constexpr uint32_t S_COL = 0;                 // NG S buffers of 64 columns; G aliases the first 32 columns of each
  constexpr uint32_t O_COL = NG * STR_ROWS;     // OUT accumulator: d <= 256 columns behind them
  // a_tmem (d <= 128): the resident operand as MMA1's A in TENSOR memory, 64 columns at the top.  MMA1 in the SS form reads
  // 4 KB of A + 2 KB of B from shared memory per K step (48 clk at 128 B/clk against a 32 clk tensor floor: ncu shows the
  // tensor pipe 66 % busy = 640 clk of MMA per ~975 clk tile); with A in tensor memory only B streams from shared memory.
  constexpr uint32_t A_COL = 448;
  const bool a_tmem = p.a_tmem != 0;
  const int a_groups = a_tmem ? (p.d + 31) / 32 : 0;      // epilogue groups that copy 16 columns (= 32 bf16) each

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_res);
    tma_prefetch_desc(&tm_str);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < MAX_STR; ++s) {
      mbar_init(&str_full[s], 1);
      mbar_init(&str_empty[s], 1);
    }
    mbar_init(res_full, 1);
    // a_tmem: the copying epilogue warps, not MMA1, are the readers of the resident block in shared memory
    mbar_init(res_empty, a_tmem ? 4 * a_groups : 1);
    mbar_init(a_full, a_tmem ? 4 * a_groups : 1);
    for (int b = 0; b < NG; ++b) {
      mbar_init(&s_full[b], 1);
      mbar_init(&g_full[b], 4);                 // the four warps (lane quadrants) of the group
      mbar_init(&buf_free[b], 1);
    }
    mbar_init(o_full, 1);
    mbar_init(o_empty, NUM_EPI_THREADS / 32);
    if (UPD)
      for (int b = 0; b < EPQ; ++b) {
        mbar_init(&stage_full[b], 4);
        mbar_init(&stage_free[b], 1);
      }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<TMEM_COLS>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int64_t n_jobs = p.n_res_blocks * p.chunks;

  // UPD: 768 threads start with 80 registers each; the control warpgroup (warps 0-3) and the update warpgroup hand part of
  // theirs to the epilogue warps (setmaxnreg at the top of every role branch, so that it dominates the role's code)
  if (warp == 0) {
    if (UPD) setmaxnreg_dec<KGEB_UPD_REG_CTRL>();
    // ================================ TMA producer ================================
    if (elect_one()) {
      int slot = 0;
      uint32_t phase = 0, rphase = 0;
      if (UPD && p.stagger_clk > 0) {
        // (tuning, KGEB_UPD_STAGGER: the hypothesis was that CTAs running jobs of equal length flush in lockstep -- 43 MB
        // bursts of update traffic; spreading their phases over one job period changed nothing)
        const long long t0 = clock64(), wait = (long long)blockIdx.x * p.stagger_clk;
        while (clock64() - t0 < wait) __nanosleep(100);
      }
      for (int64_t job = blockIdx.x; job < n_jobs; job += gridDim.x) {
        const int64_t rb = job % p.n_res_blocks, ch = job / p.n_res_blocks;
        mbar_wait(res_empty, rphase ^ 1);
        mbar_expect_tx(res_full, (uint32_t)(KS * RES_SLAB));
        for (int k = 0; k < KS; ++k)
          tma_load_2d(res_smem + (size_t)k * RES_SLAB, &tm_res, k * SLAB_K, (int32_t)(rb * RES_ROWS), res_full);
        rphase ^= 1;
        const int64_t u0 = ch * p.tiles_per_chunk, u1 = min(p.n_str_tiles, u0 + p.tiles_per_chunk);
        for (int64_t u = u0; u < u1; ++u) {
          mbar_wait(&str_empty[slot], phase ^ 1);
          mbar_expect_tx(&str_full[slot], (uint32_t)(KS * STR_SLAB));
          for (int k = 0; k < KS; ++k)
            tma_load_2d(str_smem + ((size_t)slot * KS + k) * STR_SLAB, &tm_str, k * SLAB_K, (int32_t)(u * STR_ROWS),
                        &str_full[slot]);
          if (++slot == NSTR) { slot = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (UPD) setmaxnreg_dec<KGEB_UPD_REG_CTRL>();
    // ================================ MMA1 issuer: S = RES * STR^T ================================
    if (elect_one()) {   // one elected thread for the whole loop: descriptors stay in uniform registers
      const uint32_t idesc1 = make_idesc(RES_ROWS, STR_ROWS, 0, 0, Elem<BF16>::kFmt);  // (K-major, K-major)
      const uint64_t dbase = make_desc(0, 16, 1024);
      const uint32_t tbase = tmem_base;
      int slot = 0, sbuf = 0;
      uint32_t ph = 0, bph = 0, rphase = 0;     // bph: bit b = phase of buf_free[b]
      const uint32_t res0 = smem_s, str0 = smem_s + (uint32_t)(KS * RES_SLAB);
      for (int64_t job = blockIdx.x; job < n_jobs; job += gridDim.x) {
        const int64_t ch = job / p.n_res_blocks;
        const int64_t u0 = ch * p.tiles_per_chunk, u1 = min(p.n_str_tiles, u0 + p.tiles_per_chunk);
        mbar_wait(a_tmem ? a_full : res_full, rphase);
        rphase ^= 1;
        for (int64_t u = u0; u < u1; ++u) {
          mbar_wait(&str_full[slot], ph);
          mbar_wait(&buf_free[sbuf], ((bph >> sbuf) & 1u) ^ 1u);   // MMA2 of tile u - NG has consumed this buffer's G
          tc_fence_after();
          const uint32_t acc = tbase + S_COL + (uint32_t)(sbuf * STR_ROWS);
          if (a_tmem) {
            for (int k = 0; k < KS; ++k) {
              const uint64_t sa = dbase + (uint64_t)((str0 + (uint32_t)(slot * KS + k) * STR_SLAB) >> 4);
#pragma unroll
              for (int kk = 0; kk < SLAB_K / UMMA_K; ++kk)   // A: 8 columns (16 bf16) per K step; B: +32 B per K step
                umma_ts_bf16(acc, tbase + A_COL + (uint32_t)((k * SLAB_K + kk * UMMA_K) / 2), sa + 2 * kk, idesc1,
                             (k | kk) != 0);
            }
          } else {
            for (int k = 0; k < KS; ++k) {
              const uint64_t ra = dbase + (uint64_t)((res0 + (uint32_t)k * RES_SLAB) >> 4);
              const uint64_t sa = dbase + (uint64_t)((str0 + (uint32_t)(slot * KS + k) * STR_SLAB) >> 4);
#pragma unroll
              for (int kk = 0; kk < SLAB_K / UMMA_K; ++kk)   // +32 B (= 2 in descriptor units) per K step
                umma<BF16>(acc, ra + 2 * kk, sa + 2 * kk, idesc1, (k | kk) != 0);
            }
          }
          umma_commit(&s_full[sbuf]);
          bph ^= 1u << sbuf;
          if (++sbuf == NG) sbuf = 0;
          if (++slot == NSTR) { slot = 0; ph ^= 1; }
        }
        if (!a_tmem) umma_commit(res_empty);   // all MMA1 of the job issued before this commit have read the resident block
      }
    }
  } else if (warp == 2) {
    if (UPD) setmaxnreg_dec<KGEB_UPD_REG_CTRL>();
  } else if (warp == 3) {
    if (UPD) setmaxnreg_dec<KGEB_UPD_REG_CTRL>();
    // ================================ MMA2 issuer: OUT += G * STR  (A = G from tensor memory) ================================
    if (elect_one()) {
      const uint32_t idesc2 = make_idesc(RES_ROWS, p.d, 0, 1, Elem<BF16>::kFmt);       // (K-major, MN-major)
      const uint64_t bbase = make_desc(0, STR_SLAB, 1024);
      const uint32_t tbase = tmem_base;
      int slot = 0, gbuf = 0;
      uint32_t gph = 0, ophase = 0;             // gph: bit b = phase of g_full[b]
      const uint32_t str0 = smem_s + (uint32_t)(KS * RES_SLAB);
      const uint32_t acc = tbase + O_COL;
      for (int64_t job = blockIdx.x; job < n_jobs; job += gridDim.x) {
        const int64_t ch = job / p.n_res_blocks;
        const int64_t u0 = ch * p.tiles_per_chunk, u1 = min(p.n_str_tiles, u0 + p.tiles_per_chunk);
        mbar_wait(o_empty, ophase ^ 1);  // previous job's accumulator has been flushed
        for (int64_t u = u0; u < u1; ++u) {
          mbar_wait(&g_full[gbuf], (gph >> gbuf) & 1u);
          tc_fence_after();
          const uint32_t ga = tbase + S_COL + (uint32_t)(gbuf * STR_ROWS);   // G: 64 bf16 per row = 32 columns
          const uint32_t sa = str0 + (uint32_t)(slot * KS) * STR_SLAB;
#pragma unroll
          for (int km = 0; km < STR_ROWS / UMMA_K; ++km) {
            // B: the STR tile MN-major -- UMMA_K K-rows of 128 B (8-row groups 1024 B apart = SBO); N chunks of one
            //    128 B row (SLAB_K columns) are one slab apart (LBO = STR_SLAB).
            const uint64_t bd = bbase + (uint64_t)((sa + km * UMMA_K * 128) >> 4);
            umma_ts_bf16(acc, ga + (uint32_t)(km * (UMMA_K / 2)), bd, idesc2, !(u == u0 && km == 0));
          }
          umma_commit(&str_empty[slot]);  // streamed tile free once MMA2 has read it (MMA1 of it finished long ago)
          umma_commit(&buf_free[gbuf]);
          gph ^= 1u << gbuf;
          if (++gbuf == NG) gbuf = 0;
          if (++slot == NSTR) slot = 0;
        }
        umma_commit(o_full);      // accumulator complete
        ophase ^= 1;
      }
    }
  } else if (UPD && warp >= 4 + 4 * EPQ) {
    // ================================ update warp of column part `part` ================================
    // Adagrad on the gradient box the part's epilogue warps staged in shared memory (128 rows x 32 columns, 128-byte
    // swizzle): a warp instruction covers 4 rows x 128 contiguous bytes of W / state.  Runs beside the next job's tiles:
    // measured inside the epilogue warps (which the MUFU-bound tile loop needs), the same code added 1.6 ms to a 4.0 ms kernel.
    if (KGEB_UPD_REG_UPD >= 80) setmaxnreg_inc<KGEB_UPD_REG_UPD>(); else setmaxnreg_dec<KGEB_UPD_REG_UPD>();
    const int part = warp - (4 + 4 * EPQ);
    const int sub = lane >> 3, ck = lane & 7;   // row within a group of 4, 16-byte chunk of the 128-byte box row
    const bool live = p.upd_skip == nullptr || __ldg(p.upd_skip) == 0;
    // the rate of this launch (device word of the _sched entry or the by-value parameter), read once at role start and kept
    // in shared memory behind the slot arrays: held in a register across the loop below it made ptxas spill 20-28 more
    // bytes in this kernel (-Xptxas -v); read from here the register and spill counts are those of the by-value kernel
    float* clr_s = reinterpret_cast<float*>(slot_s + EPQ * RES_ROWS);
    if (lane == 0) *clr_s = p.upd_clr_dev ? __ldg(p.upd_clr_dev) : p.upd_clr;   // (every update warp stores the same value)
    __syncwarp();
    const int nbox = (p.d + 31) / 32;
    uint8_t* stage = stage_smem + (size_t)part * STAGE_BYTES;
    uint32_t fphase = 0;
    for (int64_t job = blockIdx.x; job < n_jobs; job += gridDim.x) {
      const int64_t rb = job % p.n_res_blocks;
      for (int box = part; box < nbox; box += EPQ) {
        mbar_wait(&stage_full[part], fphase);
        fphase ^= 1;
        const int col = box * 32 + ck * 4;
        if (live && col < p.d && !(p.upd_debug & 16)) {
#pragma unroll 1
          for (int it = 0; it < 4; ++it) {
            // 8 rows per round: 16 loads of 16 bytes in flight per lane (the warp has ~16 us per box and pays ~1 us of
            // latency per round); the gradient and the slot are re-read from shared memory where they are consumed
            float4 w8[8], s8[8];
            const int r0 = it * 32 + sub;                                  // rows r0 + 4 i of the box
            const size_t base = ((size_t)rb * RES_ROWS + r0) * p.d + col;  // element offset of row r0
            const int64_t left = p.n_res - (rb * RES_ROWS + r0);           // row r0 + 4 i exists iff 4 i < left
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int sl = 4 * i < left ? slot_s[part * RES_ROWS + r0 + 4 * i] : -2;
              if (sl == -1 && !(p.upd_debug & 1)) {
                w8[i] = *reinterpret_cast<const float4*>(p.upd_w + base + (size_t)(4 * i) * p.d);
                s8[i] = *reinterpret_cast<const float4*>(p.upd_state + base + (size_t)(4 * i) * p.d);
              } else {
                w8[i] = s8[i] = make_float4(1.f, 1.f, 1.f, 1.f);
              }
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int r = r0 + 4 * i;
              const int sl = 4 * i < left ? slot_s[part * RES_ROWS + r] : -2;
              if (sl == -2) continue;
              const float4 g = *reinterpret_cast<const float4*>(stage + (size_t)r * 128 + ((ck ^ (r & 7)) << 4));
              if (sl >= 0) {
                *reinterpret_cast<float4*>(p.upd_gbuf + (size_t)sl * p.d + col) = g;
                continue;
              }
              // Adagrad with MUFU square root and reciprocal (sqrt.approx, rcp.approx: the update term is within ~3 ulp of
              // adagrad_dense_kernel's IEEE sqrt / division, i.e. ~1e-7 * |dw|).  The IEEE sequences are ~45 instructions
              // per element; this warp shares its scheduler with four epilogue warps that already use ~80 % of the issue
              // slots, and with them the update warp fell behind the tile pipeline (kernel 5.7 instead of 4.1 ms).
              float4 w = w8[i], st = s8[i];
              const float clr = *clr_s;
              st.x = fmaf(g.x, g.x, st.x); st.y = fmaf(g.y, g.y, st.y); st.z = fmaf(g.z, g.z, st.z); st.w = fmaf(g.w, g.w, st.w);
              w.x = fmaf(-clr * g.x, rcp_approx(sqrt_approx(st.x) + p.upd_eps), w.x);
              w.y = fmaf(-clr * g.y, rcp_approx(sqrt_approx(st.y) + p.upd_eps), w.y);
              w.z = fmaf(-clr * g.z, rcp_approx(sqrt_approx(st.z) + p.upd_eps), w.z);
              w.w = fmaf(-clr * g.w, rcp_approx(sqrt_approx(st.w) + p.upd_eps), w.w);
              if (p.upd_debug & 2) continue;
              const size_t off = base + (size_t)(4 * i) * p.d;
              *reinterpret_cast<float4*>(p.upd_w + off) = w;
              *reinterpret_cast<float4*>(p.upd_state + off) = st;
              uint2 mb;
              asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(mb.x) : "f"(w.y), "f"(w.x));
              asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(mb.y) : "f"(w.w), "f"(w.z));
              *reinterpret_cast<uint2*>(p.upd_mirror + off) = mb;
            }
          }
        }
        mbar_arrive_warp(&stage_free[part]);      // (all lanes have read the staging box and the slots: __syncwarp inside)
      }
    }
  } else if (warp >= 4) {
    if (UPD) setmaxnreg_inc<KGEB_UPD_REG_EPI>();
    // ================================ epilogue ================================
    const int ew = warp - 4;
    const int quad = ew & 3;                               // == warp % 4 : TMEM lane quadrant this warp may access
    const int part = ew >> 2;                              // group 0..NG-1 = buffer / tile residue served by this warp
    const int trow = quad * 32 + lane;                     // resident row (TMEM lane) of this thread
    const uint32_t lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16);
    const uint32_t buf_addr = lane_addr + S_COL + (uint32_t)(part * STR_ROWS);
    uint32_t sph = 0, ophase = 0, aphase = 0, uphase = 0;
    int64_t gunit = 0;                                     // global tile counter (buffers rotate across jobs too)
    for (int64_t job = blockIdx.x; job < n_jobs; job += gridDim.x) {
      const int64_t rb = job % p.n_res_blocks, ch = job / p.n_res_blocks;
      const int64_t u0 = ch * p.tiles_per_chunk, u1 = min(p.n_str_tiles, u0 + p.tiles_per_chunk);
      const int64_t res_row = rb * RES_ROWS + trow;
      EpiRow er;
      if (FLASH) {
        if (res_row < p.B) er.fl_m2 = -p.mref[res_row] * 1.4426950408889634f;
      } else if (RES_IS_Q && res_row < p.B) {
        er.my_rs = p.inv_batch * (HAS_RS ? p.row_scale[res_row] : 1.f);
        if (LOSS == KGEB_LOSS_KL) er.my_lse = p.lse[res_row];
      }
      int upd_slot = 0;
      if (UPD && res_row < p.n_res) {
        // fused update: the slot of this thread's row (consumed at the flush: the load stays in flight under the job), and
        // the row's lines of W and of the Adagrad state pulled into L2 -- they are wanted ~15 us from now
        upd_slot = __ldg(p.upd_slot + res_row);
        if (!(p.upd_debug & 8))
        for (int box = part; box * 32 < p.d; box += EPQ) {
          asm volatile("prefetch.global.L2 [%0];" ::"l"(p.upd_w + (size_t)res_row * p.d + box * 32));
          asm volatile("prefetch.global.L2 [%0];" ::"l"(p.upd_state + (size_t)res_row * p.d + box * 32));
        }
      }
      if (a_tmem && part < a_groups) {
        // resident block: shared memory (TMA, 128-byte swizzle) -> tensor memory columns [A_COL + 16 part, + 16) of this
        // thread's lane: 32 bf16 = bytes [64 part, 64 part + 64) of the row = four 16-byte chunks of slab part / 2.
        // (Every MMA of the previous job has completed: this warp passed o_full.)
        mbar_wait(res_full, aphase);
        const uint32_t rowa = smem_s + (uint32_t)((part >> 1) * RES_SLAB + trow * 128);
        uint32_t w[16];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int ck = (part & 1) * 4 + c;
          asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                       : "=r"(w[4 * c]), "=r"(w[4 * c + 1]), "=r"(w[4 * c + 2]), "=r"(w[4 * c + 3])
                       : "r"(rowa + (uint32_t)((ck ^ (trow & 7)) << 4)));
        }
        tmem_st16(lane_addr + A_COL + (uint32_t)(16 * part), w);
        tmem_wait_st();
        tc_fence_before();
        mbar_arrive_warp(a_full);
        mbar_arrive_warp(res_empty);      // the producer may prefetch the next job's block
      }
      aphase ^= 1;
      // first tile of this job that belongs to this group
      int64_t u = u0 + (((int64_t)part - gunit) % NG + NG) % NG;
      for (; u < u1; u += NG) {
        mbar_wait(&s_full[part], sph);
        sph ^= 1;
        tc_fence_after();
        float v[COLS_PER_WARP];
#pragma unroll 1
        for (int pass = 0; pass < 2; ++pass) {
          tmem_ld32(buf_addr + (uint32_t)(pass * COLS_PER_WARP), v);
          epi_math<RES_IS_Q, LOSS, HAS_RS, STATS, FLASH>(v, p, er, u * STR_ROWS + pass * COLS_PER_WARP, lane, kc_s);
          // G of these 32 columns: 16 words of two bf16 -> columns [16 pass, 16 pass + 16) of the same buffer.  All 64 S
          // columns of this warp's rows are in registers / consumed before the first word of pass 1 is written
          // (pass 0 only touches columns [0, 16), which it has loaded itself).
          uint32_t w[16];
#pragma unroll
          for (int j = 0; j < 16; ++j)
            asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w[j]) : "f"(v[2 * j + 1]), "f"(v[2 * j]));
          tmem_st16(buf_addr + (uint32_t)(pass * (COLS_PER_WARP / 2)), w);
        }
        tmem_wait_st();
        tc_fence_before();
        mbar_arrive_warp(&g_full[part]);
      }
      gunit += u1 - u0;
      if (FLASH && res_row < p.B) {
        float* sp = p.stat_partial + (((size_t)ch * 4 + part) * p.B + res_row) * 2;
        const float l = ((er.fl_l[0] + er.fl_l[1]) + (er.fl_l[2] + er.fl_l[3])) - (float)er.n_pad * ex2_ftz(er.fl_m2);
        sp[0] = l;
        sp[1] = 0.f;
        // exp(x - mref) left the fp32 / bf16 range (a score > 88 nats above the reference): the caller re-runs the step
        // with the two-pass kernels (online maximum).  Finite sums are exact whatever their magnitude.
        if (!(fabsf(l) <= 3.0e38f)) *p.status = 1;
      }
      if (STATS && res_row < p.B) {
        float* sp = p.stat_partial + (((size_t)ch * 4 + part) * p.B + res_row) * 2;
        const float zp = p.offset;
        const float st_sp = fmaf(0.69314718f, er.st_lg, er.st_mx);
        sp[0] = st_sp - (float)er.n_pad * fmaf(0.69314718f, __log2f(1.f + __expf(-fabsf(zp))), fmaxf(zp, 0.f));
        sp[1] = er.st_x - (float)er.n_pad * zp;
      }
      // flush the job's accumulator
      mbar_wait(o_full, ophase);
      ophase ^= 1;
      tc_fence_after();
      bool o_released = false;
      if (RES_IS_Q) {
        for (int c0 = part * 16; c0 < p.d; c0 += 16 * EPQ) {
          float o[16];
          tmem_ld16(lane_addr + O_COL + (uint32_t)c0, o);
          if (res_row < p.n_res) {
            float* dst = p.out + ((size_t)ch * p.B + res_row) * p.d + c0;
            float big = 0.f;
#pragma unroll
            for (int c = 0; c < 16; c += 4) {
              *reinterpret_cast<float4*>(dst + c) = make_float4(o[c], o[c + 1], o[c + 2], o[c + 3]);
              if (FLASH) big = fmaxf(fmaxf(big, fmaxf(fabsf(o[c]), fabsf(o[c + 1]))), fmaxf(fabsf(o[c + 2]), fabsf(o[c + 3])));
            }
            if (FLASH && !(big <= 3.0e38f)) *p.status = 1;   // inf or NaN in the accumulator
          }
        }
      } else if (UPD) {
        // Adagrad by the update warp of this column part: stage the accumulator box (128 rows x 32 columns) and the rows'
        // slots in shared memory and hand them over; the tensor-memory accumulator is free as soon as it has been read
        uint8_t* stage = stage_smem + (size_t)part * STAGE_BYTES;
        const int nbox = (p.d + 31) / 32;
        for (int box = part; box < nbox; box += EPQ) {
          mbar_wait(&stage_free[part], uphase ^ 1);      // the update warp is done with the previous box
          uphase ^= 1;
          slot_s[part * RES_ROWS + trow] = upd_slot;
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            float o[16];
            tmem_ld16(lane_addr + O_COL + (uint32_t)(box * 32 + h * 16), o);
            uint8_t* rowp = stage + (size_t)trow * 128;
#pragma unroll
            for (int j = 0; j < 4; ++j)
              *reinterpret_cast<float4*>(rowp + (((h * 4 + j) ^ (trow & 7)) << 4)) =
                  make_float4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
          }
          mbar_arrive_warp(&stage_full[part]);
          if (box + EPQ >= nbox) {     // the accumulator has been read: MMA2 of the next job may start
            tc_fence_before();
            mbar_arrive_warp(o_empty);
            o_released = true;
          }
        }
      } else {
        uint8_t* stage = stage_smem + (size_t)part * STAGE_BYTES;
        const bool leader = (quad == 0 && lane == 0);
        const int nbox = (p.d + 31) / 32;
        for (int box = part; box < nbox; box += EPQ) {
          if (leader) bulk_wait_read0();             // the previous store from this staging box has read it
          named_bar_sync(1 + part, 128);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            float o[16];
            tmem_ld16(lane_addr + O_COL + (uint32_t)(box * 32 + h * 16), o);
            uint8_t* rowp = stage + (size_t)trow * 128;
#pragma unroll
            for (int j = 0; j < 4; ++j)
              *reinterpret_cast<float4*>(rowp + (((h * 4 + j) ^ (trow & 7)) << 4)) =
                  make_float4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
          }
          fence_proxy_async();
          named_bar_sync(1 + part, 128);
          if (leader) {
            if (p.overwrite) tma_store_2d(&tm_out, stage, box * 32, (int32_t)(rb * RES_ROWS));
            else tma_reduce_add_2d(&tm_out, stage, box * 32, (int32_t)(rb * RES_ROWS));
            bulk_commit();
          }
        }
      }
      if (!o_released) {
        tc_fence_before();
        mbar_arrive_warp(o_empty);
      }
    }
  }

  if (!RES_IS_Q && warp >= 4 && ((warp - 4) & 3) == 0 && lane == 0) bulk_wait0();  // outstanding TMA stores / reduce-adds
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------------
// exact fp32 sparse label part (entry-parallel: hot rows / hot entities cost no more than cold ones)
// ---------------------------------------------------------------------------------------------
__global__ void reduce_dq_partials_kernel(const float* __restrict__ partial, int64_t chunks, int64_t numel,
                                          const float* __restrict__ label_part, float* __restrict__ dQ) {
  int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) * 4;
  for (; i < numel; i += (int64_t)gridDim.x * blockDim.x * 4) {   // numel = B*d with d % 16 == 0
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int64_t k = 0; k < chunks; ++k) {  // fixed order
      const float4 v = *reinterpret_cast<const float4*>(partial + k * numel + i);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    if (label_part) {   // exact fp32 label rows, summed per query row on the side stream
      const float4 v = *reinterpret_cast<const float4*>(label_part + i);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    *reinterpret_cast<float4*>(dQ + i) = s;
  }
}

// Label entries i (entries [lab_off[B], nnz) are padding of a fixed-size label buffer); one warp handles
// LABEL_EPW consecutive entries:
//   rows_dq[i,:] = -w_q * table[e,:]   (summed per query row q ; keys erow[] are ascending)
//   rows_dt[i,:] = -w_q * Q[q,:]       (scattered into dTable[e,:] ; keys ent[])
// with w_q = tscale[q] * inv_batch * row_scale[q]; entries outside this shard get zero rows.
// The row of the warp's first entry comes from a 32-ary search over lab_off (3 dependent loads for B = 4096 instead
// of the 12 of a binary search -- this kernel is pure latency), the following entries walk forward from it.
constexpr int LABEL_EPW = 4;
__global__ void __launch_bounds__(256)
label_entry_rows_kernel(const float* __restrict__ Q, const float* __restrict__ table, int64_t B, int d, int64_t e_lo,
                        int64_t n_ent, const int64_t* __restrict__ lab_off, const int64_t* __restrict__ lab_col,
                        const float* __restrict__ tscale, const float* __restrict__ row_scale, float inv_batch, int64_t nnz,
                        float* __restrict__ rows_dq, float* __restrict__ rows_dt, int64_t* __restrict__ ent,
                        int64_t* __restrict__ erow, float* __restrict__ entry_dot, float add_per_entry) {
  const int lane = threadIdx.x & 31;
  const int64_t i0 = (blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5)) * LABEL_EPW;
  if (i0 >= nnz) return;
  const int64_t n_real = lab_off[B];
  // last q in [0, B] with lab_off[q] <= i0 (lab_off[0] = 0 <= i0 always)
  int64_t lo = 0, hi = B;
  while (lo < hi) {
    const int64_t step = (hi - lo + 32) / 32;          // ceil((hi - lo + 1) / 32)
    const int64_t probe = lo + (int64_t)lane * step;
    const bool ok = probe <= hi && lab_off[probe] <= i0;
    const unsigned m = __ballot_sync(0xffffffffu, ok);  // lane 0 always votes yes
    const int top = 31 - __clz((int)m);
    const int64_t nlo = lo + (int64_t)top * step;
    hi = min(hi, nlo + step - 1);
    lo = nlo;
  }
  int64_t q = lo;
#pragma unroll 1
  for (int k = 0; k < LABEL_EPW; ++k) {
    const int64_t i = i0 + k;
    if (i >= nnz) break;
    const bool real = i < n_real;
    if (real) while (q < B - 1 && lab_off[q + 1] <= i) ++q;   // skips empty rows
    int64_t e = 0;
    float w = 0.f;
    bool in_shard = false;
    if (real) {
      e = lab_col[i] - e_lo;
      in_shard = (e >= 0 && e < n_ent);
      if (in_shard) w = tscale ? tscale[q] * inv_batch * (row_scale ? row_scale[q] : 1.f) : 0.f;
      else e = e < 0 ? 0 : n_ent - 1;   // zero row; the monotone clamp keeps ent[] in the order of lab_col (lab_perm)
    }
    const int64_t qq = real ? q : 0;
    float dot = 0.f;
    for (int c = lane * 4; c < d; c += 128) {   // d % 4 == 0
      const float4 tv = __ldg(reinterpret_cast<const float4*>(table + e * d + c));
      const float4 qv = *reinterpret_cast<const float4*>(Q + qq * d + c);
      dot = fmaf(qv.x, tv.x, fmaf(qv.y, tv.y, fmaf(qv.z, tv.z, fmaf(qv.w, tv.w, dot))));
      if (rows_dq) *reinterpret_cast<float4*>(rows_dq + i * d + c) = make_float4(-w * tv.x, -w * tv.y, -w * tv.z, -w * tv.w);
      if (rows_dt) *reinterpret_cast<float4*>(rows_dt + i * d + c) = make_float4(-w * qv.x, -w * qv.y, -w * qv.z, -w * qv.w);
    }
    if (entry_dot) dot = warp_sum(dot);   // warp-uniform branch
    if (lane == 0) {
      ent[i] = e;
      erow[i] = qq;
      if (entry_dot) entry_dot[i] = in_shard ? dot + add_per_entry : 0.f;   // x_ij (+offset) at the label, in-shard only
    }
  }
}

struct Plan {
  Params p;
  size_t smem;
};

// v2 pipeline (tc_bwd4_kernel) unless KGEB_BWD_V2=0 in the environment (the two-buffer kernel stays for A/B timing)
static bool use_v2() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("KGEB_BWD_V2");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}

static Plan make_plan(bool res_is_q, bool bf16, int64_t B, int d, int64_t n_ent) {
  Plan pl;
  Params& p = pl.p;
  memset(&p, 0, sizeof(p));
  const int slab_k = bf16 ? 64 : 32;
  p.B = B;
  p.d = d;
  p.ks = (d + slab_k - 1) / slab_k;
  p.n_res = res_is_q ? B : n_ent;
  p.n_str = res_is_q ? n_ent : B;
  p.n_res_blocks = (p.n_res + RES_ROWS - 1) / RES_ROWS;
  p.n_str_tiles = (p.n_str + STR_ROWS - 1) / STR_ROWS;
  if (res_is_q) {
    int64_t chunks = kNumSMs / (p.n_res_blocks > 0 ? p.n_res_blocks : 1);
    if (chunks < 1) chunks = 1;
    if (chunks > p.n_str_tiles) chunks = p.n_str_tiles > 0 ? p.n_str_tiles : 1;
    p.tiles_per_chunk = (p.n_str_tiles + chunks - 1) / chunks;
    if (p.tiles_per_chunk < 1) p.tiles_per_chunk = 1;
    p.chunks = (p.n_str_tiles + p.tiles_per_chunk - 1) / p.tiles_per_chunk;
    if (p.chunks < 1) p.chunks = 1;
  } else {
    p.chunks = 1;
    p.tiles_per_chunk = p.n_str_tiles > 0 ? p.n_str_tiles : 1;
  }
  // barriers / tensor-memory slot (512 B) + 1 KiB alignment slack; v2 dTable kernel: + the per-query exponent offsets of
  // all streamed rows (KL; up to 4096 rows -- larger batches use the shuffle path)
  const int64_t colk_n = (!res_is_q && use_v2() && bf16 && B <= 4096) ? ((B + 63) / 64) * 64 : 0;
  p.colk_n = (int)colk_n;
  p.colk_n_alloc = (int)colk_n;
  // (+ 2 KiB: the touched-row slots of the tile, one copy per column part, for the fused update; + 16 B: its learning rate)
  const size_t fixed = 1024 + 512 + (size_t)colk_n * 4 + (res_is_q ? 0 : (size_t)EPQ * RES_ROWS * 4 + 16);
  const size_t g_bytes = (use_v2() && bf16) ? 0 : (size_t)(STR_ROWS / slab_k) * RES_SLAB;   // v2: G lives in tensor memory
  const size_t base = (size_t)p.ks * RES_SLAB + 2 * g_bytes + (res_is_q ? 0 : (size_t)EPQ * STAGE_BYTES);
  int nstr = (int)((SMEM_BUDGET - fixed - base) / ((size_t)p.ks * STR_SLAB));
  if (nstr > MAX_STR) nstr = MAX_STR;
  p.nstr = nstr;
  pl.smem = base + (size_t)nstr * p.ks * STR_SLAB + fixed;
  p.a_tmem = (use_v2() && bf16 && d <= 128 && !getenv("KGEB_NO_A_TMEM")) ? 1 : 0;
  return pl;
}

template <bool RES_IS_Q>
static int launch_bwd(const Plan& pl, const CUtensorMap& m_res, const CUtensorMap& m_str, const CUtensorMap& m_out,
                      int64_t jobs, cudaStream_t st, bool flash = false) {
  const int grid = (int)(jobs < kNumSMs ? jobs : kNumSMs);
  cudaError_t e = cudaSuccess;
  // (A raised launch priority for this kernel was tried and measured worse: it starts a few microseconds earlier but
  // then starves the label kernels of the other stream, which the second tile kernel waits for.)
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(NUM_THREADS);
  cfg.dynamicSmemBytes = pl.smem;
  cfg.stream = st;
  cfg.attrs = nullptr;
  cfg.numAttrs = 0;
#define KGEB_BWD_LAUNCH(LOSS_, RS_, ST_)                                                                              \
  {                                                                                                                   \
    e = cudaFuncSetAttribute(tc_bwd_kernel<RES_IS_Q, true, LOSS_, RS_, ST_>,                                          \
                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem);                              \
    if (e != cudaSuccess) return cuda_status(e, "tc_bwd smem attribute");                                             \
    e = cudaLaunchKernelEx(&cfg, tc_bwd_kernel<RES_IS_Q, true, LOSS_, RS_, ST_>, m_res, m_str, m_out, pl.p);           \
    if (e != cudaSuccess) return cuda_status(e, "tc_bwd launch");                                                     \
  }
  const bool rs = pl.p.row_scale != nullptr;
  const bool stats = RES_IS_Q && pl.p.stat_partial != nullptr && pl.p.loss == KGEB_LOSS_BCE;
  if (use_v2()) {
#define KGEB_BWD4_LAUNCH(LOSS_, RS_, ST_, FL_)                                                                        \
  {                                                                                                                   \
    e = cudaFuncSetAttribute(tc_bwd4_kernel<RES_IS_Q, LOSS_, RS_, ST_, FL_>,                                          \
                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem);                              \
    if (e != cudaSuccess) return cuda_status(e, "tc_bwd4 smem attribute");                                            \
    e = cudaLaunchKernelEx(&cfg, tc_bwd4_kernel<RES_IS_Q, LOSS_, RS_, ST_, FL_>, m_res, m_str, m_out, pl.p);           \
    if (e != cudaSuccess) return cuda_status(e, "tc_bwd4 launch");                                                    \
  }
    if (!RES_IS_Q && pl.p.upd_w != nullptr) {
      cfg.blockDim = dim3(NUM_THREADS + UPD_THREADS);
#define KGEB_UPD_LAUNCH(LOSS_, RS_)                                                                                   \
  {                                                                                                                   \
    e = cudaFuncSetAttribute(tc_bwd4_kernel<false, LOSS_, RS_, false, false, true>,                                   \
                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem);                              \
    if (e != cudaSuccess) return cuda_status(e, "tc_bwd4 smem attribute");                                            \
    e = cudaLaunchKernelEx(&cfg, tc_bwd4_kernel<false, LOSS_, RS_, false, false, true>, m_res, m_str, m_out, pl.p);    \
    if (e != cudaSuccess) return cuda_status(e, "tc_bwd4 launch");                                                    \
  }
      if (pl.p.loss == KGEB_LOSS_KL) {
        if (rs) KGEB_UPD_LAUNCH(KGEB_LOSS_KL, true) else KGEB_UPD_LAUNCH(KGEB_LOSS_KL, false)
      } else {
        if (rs) KGEB_UPD_LAUNCH(KGEB_LOSS_BCE, true) else KGEB_UPD_LAUNCH(KGEB_LOSS_BCE, false)
      }
#undef KGEB_UPD_LAUNCH
    } else if (flash) {
      KGEB_BWD4_LAUNCH(KGEB_LOSS_KL, false, false, RES_IS_Q)
    } else if (pl.p.loss == KGEB_LOSS_KL) {
      if (rs) KGEB_BWD4_LAUNCH(KGEB_LOSS_KL, true, false, false) else KGEB_BWD4_LAUNCH(KGEB_LOSS_KL, false, false, false)
    } else if (stats) {
      if (rs) KGEB_BWD4_LAUNCH(KGEB_LOSS_BCE, true, RES_IS_Q, false) else KGEB_BWD4_LAUNCH(KGEB_LOSS_BCE, false, RES_IS_Q, false)
    } else {
      if (rs) KGEB_BWD4_LAUNCH(KGEB_LOSS_BCE, true, false, false) else KGEB_BWD4_LAUNCH(KGEB_LOSS_BCE, false, false, false)
    }
#undef KGEB_BWD4_LAUNCH
    KGEB_LAUNCH_CHECK("tc_bwd4_kernel");
    return KGEB_OK;
  }
  if (flash) {
    if (RES_IS_Q) {
      e = cudaFuncSetAttribute(tc_bwd_kernel<RES_IS_Q, true, KGEB_LOSS_KL, false, false, RES_IS_Q>,
                               cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem);
      if (e != cudaSuccess) return cuda_status(e, "tc_bwd smem attribute");
      e = cudaLaunchKernelEx(&cfg, tc_bwd_kernel<RES_IS_Q, true, KGEB_LOSS_KL, false, false, RES_IS_Q>, m_res, m_str, m_out, pl.p);
      if (e != cudaSuccess) return cuda_status(e, "tc_bwd launch");
    }
  } else if (pl.p.loss == KGEB_LOSS_KL) {
    if (rs) KGEB_BWD_LAUNCH(KGEB_LOSS_KL, true, false) else KGEB_BWD_LAUNCH(KGEB_LOSS_KL, false, false)
  } else if (stats) {
    if (rs) KGEB_BWD_LAUNCH(KGEB_LOSS_BCE, true, RES_IS_Q) else KGEB_BWD_LAUNCH(KGEB_LOSS_BCE, false, RES_IS_Q)
  } else {
    if (rs) KGEB_BWD_LAUNCH(KGEB_LOSS_BCE, true, false) else KGEB_BWD_LAUNCH(KGEB_LOSS_BCE, false, false)
  }
#undef KGEB_BWD_LAUNCH
  KGEB_LAUNCH_CHECK("tc_bwd_kernel");
  return KGEB_OK;
}

// colk[q] = (log(inv_batch * row_scale[q]) - lse[q]) * log2(e) for q < B, 0 for the padding up to n (KL dTable kernel)
__global__ void colk_kernel(const float* __restrict__ lse, const float* __restrict__ row_scale, float inv_batch, int64_t B,
                            int n, float* __restrict__ colk) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float v = 0.f;
  if (i < B) v = (__logf(inv_batch * (row_scale ? row_scale[i] : 1.f)) - lse[i]) * 1.4426950408889634f;
  colk[i] = v;
}

// rowstat[r] = (sum softplus, 0, sum (x+off), label_dot[r]) from the per-(chunk, column part) partials, fixed order
__global__ void reduce_stat_partials_kernel(const float* __restrict__ sp, int64_t chunks, int64_t B,
                                            const float* __restrict__ label_dot, float* __restrict__ rowstat) {
  const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (r >= B) return;
  float a = 0.f, b = 0.f;
  for (int64_t k = 0; k < chunks * 4; ++k) {
    a += sp[(k * B + r) * 2];
    b += sp[(k * B + r) * 2 + 1];
  }
  float* o = rowstat + r * 4;
  o[0] = a; o[1] = 0.f; o[2] = b; o[3] = label_dot[r];
}

__global__ void __launch_bounds__(256)
label_row_sum2_kernel(const float* __restrict__ entry_dot, const int64_t* __restrict__ lab_off, int64_t B,
                      float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t r = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= B) return;
  float acc = 0.f;
  for (int64_t i = lab_off[r] + lane; i < lab_off[r + 1]; i += 32) acc += entry_dot[i];
  acc = warp_sum(acc);
  if (lane == 0) out[r] = acc;
}

__global__ void to_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int64_t n) {
  int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) * 4;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x * 4;
  for (; i + 3 < n; i += stride) {
    float4 v = *reinterpret_cast<const float4*>(src + i);
    __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    uint2 o;
    o.x = *reinterpret_cast<uint32_t*>(&a);
    o.y = *reinterpret_cast<uint32_t*>(&b);
    *reinterpret_cast<uint2*>(dst + i) = o;
  }
  if (i < n) for (int64_t j = i; j < n; ++j) dst[j] = __float2bfloat16_rn(src[j]);
}

// FLASH reference score of row q (fp32):
//   mref[q] = max( max over a strided sample of <= 64 entities of the shard + min(2 sigma, 40),
//                  max over <= 192 of THIS BATCH's label entities (strided over lab_col, those inside the shard),
//                  the largest score among the row's own labels )
// exp(x - mref) must stay inside the fp32 / bf16 range for every entity: x - mref < ~88 nats.  The strided sample centres
// the window for bell-shaped rows (the shard maximum lies ~3 sigma above the maximum of 64 samples); the label entities
// are where a trained model puts its large scores -- the row's own answers, and the popular answers that recur in every
// batch and carry the largest norms.  This is a heuristic: the kernel reports rows it failed on (Params::status) and the
// caller repeats the step with the two-pass kernels, so a wrong guess costs time, never a wrong result.
// One warp per row, four candidate rows in flight per iteration (the loop is pure L2 latency otherwise).
// (16 warps: the candidate loop is a chain of dependent L2 loads and shuffle reductions, ~1 us per candidate and warp; with 4
// warps per block the kernel took 65 us whatever the shard size -- 5 % of a step at 8 GPUs)
constexpr int kFlashSamples = 64, kFlashLabelSamples = 192, kFlashWarps = 16, kFlashRows = 8;
__global__ void __launch_bounds__(kFlashWarps * 32)
sample_max_kernel(const float* __restrict__ Q, const float* __restrict__ table, int64_t B, int d, int64_t e_lo, int64_t n_ent,
                  const int64_t* __restrict__ lab_off, const int64_t* __restrict__ lab_col, const float* __restrict__ entry_dot,
                  float* __restrict__ mref) {
  // A block scores kFlashRows query rows against the (row-independent) candidate list: every candidate row is read once
  // per block and dotted with all of the block's query rows (one candidate per warp at a time, lanes over the dimension).
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t r0 = blockIdx.x * (int64_t)kFlashRows;
  __shared__ float s_q[kFlashRows][256];
  __shared__ float s_best[kFlashWarps][kFlashRows], s_lab[kFlashWarps][kFlashRows], s_sum[kFlashWarps][kFlashRows],
      s_sum2[kFlashWarps][kFlashRows];
  for (int i = threadIdx.x; i < kFlashRows * 256; i += blockDim.x) {
    const int rr = i >> 8, c = i & 255;
    s_q[rr][c] = (r0 + rr < B && c < d) ? Q[(r0 + rr) * d + c] : 0.f;
  }
  __syncthreads();
  const int64_t ns = n_ent < kFlashSamples ? n_ent : kFlashSamples;
  const int64_t n_lab = lab_off[B];
  const int64_t nl = n_lab < kFlashLabelSamples ? n_lab : kFlashLabelSamples;
  float best[kFlashRows], blab[kFlashRows], sum[kFlashRows], sum2[kFlashRows];
#pragma unroll
  for (int rr = 0; rr < kFlashRows; ++rr) { best[rr] = -INFINITY; blab[rr] = -INFINITY; sum[rr] = 0.f; sum2[rr] = 0.f; }
  for (int64_t k = warp; k < ns + nl; k += kFlashWarps) {
    const int64_t e = k < ns ? (k * n_ent) / ns : lab_col[((k - ns) * n_lab) / nl] - e_lo;
    if (e < 0 || e >= n_ent) continue;                       // a label entity of another shard (warp-uniform)
    float t[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) t[i] = lane + 32 * i < d ? __ldg(table + e * d + lane + 32 * i) : 0.f;
#pragma unroll
    for (int rr = 0; rr < kFlashRows; ++rr) {
      float a = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) a = fmaf(s_q[rr][lane + 32 * i], t[i], a);
      const float x = warp_sum(a);
      if (k < ns) { best[rr] = fmaxf(best[rr], x); sum[rr] += x; sum2[rr] = fmaf(x, x, sum2[rr]); }
      else blab[rr] = fmaxf(blab[rr], x);
    }
  }
  if (lane == 0)
#pragma unroll
    for (int rr = 0; rr < kFlashRows; ++rr) {
      s_best[warp][rr] = best[rr]; s_lab[warp][rr] = blab[rr]; s_sum[warp][rr] = sum[rr]; s_sum2[warp][rr] = sum2[rr];
    }
  __syncthreads();
  // one warp per row finishes: combine the warps' partials (fixed order) and add the row's own label scores
  for (int rr = warp; rr < kFlashRows; rr += kFlashWarps) {
    const int64_t r = r0 + rr;
    if (r >= B) continue;
    float m_lab = -INFINITY;
    if (entry_dot)   // exact scores at the row's own labels inside this shard
      for (int64_t i = lab_off[r] + lane; i < lab_off[r + 1]; i += 32) {
        const int64_t e = lab_col[i] - e_lo;
        if (e >= 0 && e < n_ent) m_lab = fmaxf(m_lab, entry_dot[i]);
      }
    m_lab = warp_max(m_lab);
    if (lane == 0) {
      float bs = -INFINITY, sm = 0.f, sm2 = 0.f;
      for (int w = 0; w < kFlashWarps; ++w) {
        bs = fmaxf(bs, s_best[w][rr]); m_lab = fmaxf(m_lab, s_lab[w][rr]); sm += s_sum[w][rr]; sm2 += s_sum2[w][rr];
      }
      const float mean = sm / (float)ns;
      const float sigma = sqrtf(fmaxf(sm2 / (float)ns - mean * mean, 0.f));
      mref[r] = fmaxf(bs + fminf(2.f * sigma, 40.f), m_lab);
    }
  }
}

// rowstat[r] = (mref, sum_e exp(x - mref), 0, sum of x over the row's labels) -- the layout of the forward statistics
__global__ void flash_rowstat_kernel(const float* __restrict__ sp, int64_t chunks, int64_t B, const float* __restrict__ mref,
                                     const float* __restrict__ label_dot, float* __restrict__ rowstat) {
  const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (r >= B) return;
  float l = 0.f;
  for (int64_t k = 0; k < chunks * 4; ++k) l += sp[(k * B + r) * 2];     // fixed order
  float* o = rowstat + r * 4;
  o[0] = mref ? mref[r] : -INFINITY; o[1] = l; o[2] = 0.f; o[3] = label_dot[r];
}

// dQ[r,:] = w_r * exp(mref_r - lse_r) * o_sum[r,:] + label rows,  w_r = inv_batch * row_scale[r] * (row r has labels)
__global__ void flash_dq_kernel(const float* __restrict__ o_sum, const float* __restrict__ rowstat_local,
                                const float* __restrict__ lse, const int64_t* __restrict__ lab_off, float inv_batch,
                                const float* __restrict__ row_scale, const float* __restrict__ dq_lab, int64_t B, int d,
                                float* __restrict__ dQ) {
  const int64_t numel = B * d;
  int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) * 4;
  for (; i < numel; i += (int64_t)gridDim.x * blockDim.x * 4) {
    const int64_t r = i / d;
    const bool has = lab_off[r + 1] > lab_off[r];
    const float w = has ? inv_batch * (row_scale ? row_scale[r] : 1.f) * __expf(rowstat_local[r * 4] - lse[r]) : 0.f;
    const float4 o = *reinterpret_cast<const float4*>(o_sum + i);
    float4 v = make_float4(w * o.x, w * o.y, w * o.z, w * o.w);
    if (dq_lab) {
      const float4 a = *reinterpret_cast<const float4*>(dq_lab + i);
      v.x += a.x; v.y += a.y; v.z += a.z; v.w += a.w;
    }
    *reinterpret_cast<float4*>(dQ + i) = v;
  }
}

}  // namespace tcb

bool tc_bwd_supported(int math, int d) { return math == KGEB_MATH_BF16 && d % 16 == 0 && d <= 256; }

int tc_to_bf16(const float* src, void* dst, int64_t n, cudaStream_t st) {
  if (n == 0) return KGEB_OK;
  KGEB_REQUIRE(((reinterpret_cast<uintptr_t>(src) & 15) | (reinterpret_cast<uintptr_t>(dst) & 7)) == 0,
               "to_bf16: misaligned buffers");
  int64_t blocks = (n / 4 + 255) / 256 + 1;
  int grid = (int)(blocks > (int64_t)kNumSMs * 16 ? (int64_t)kNumSMs * 16 : blocks);
  tcb::to_bf16_kernel<<<grid, 256, 0, st>>>(src, reinterpret_cast<__nv_bfloat16*>(dst), n);
  KGEB_LAUNCH_CHECK("to_bf16");
  return KGEB_OK;
}

}  // namespace kgeb

extern "C" int scatter_add_rows_presorted(const int64_t* keys, const float* rows, int64_t n, int d, float* dense,
                                          int64_t vocab, void* workspace, int64_t workspace_bytes, cudaStream_t st);

namespace kgeb {

static int64_t a256(int64_t x) { return (x + 255) / 256 * 256; }

int64_t tc_bwd_workspace_bytes(int64_t B, int d, int64_t n_ent, int64_t nnz) {
  if (nnz < 1) nnz = 1;
  return a256((int64_t)kNumSMs * B * d * 4) + a256(B * (int64_t)d * 4) + 2 * a256(nnz * (int64_t)d * 4) + 2 * a256(nnz * 8) +
         a256((int64_t)kNumSMs * 4 * B * 2 * 4) + a256(nnz * 4) + 2 * a256(B * 4) + kgeb_scatter_workspace_bytes(nnz, d) + 4096;
}

// A library-owned side stream per device: the sparse label part of a call is independent of its tile kernel, so it
// is forked onto the side stream and joined where its result is consumed (plain event fork / join: works in eager
// mode and inside a CUDA-graph capture, where the side stream joins the capture).
struct SideStream {
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
  cudaEvent_t tiles = nullptr;   // recorded right after the dQ tile kernel (kgeb_fused_bwd_wait_tiles)
};
// which: 0 for calls that produce dQ, 1 for dTable-only calls -- the two halves of a step are issued as two calls on
// two streams (trainer.py) and must not queue behind each other's label chains
static SideStream* side_stream(int which) {
  static thread_local SideStream per_dev[64][2];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  SideStream& s = per_dev[dev][which];
  if (!s.stream) {
    if (cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s.tiles, cudaEventDisableTiming) != cudaSuccess)
      return nullptr;
  }
  return &s;
}

// Qb / tableb: bf16 mirrors of Q [B,d] and of the table shard [n_ent,d]
int tc_fused_bwd(int loss, const float* Q, const void* Qb, int64_t B, int d, const float* table, const void* tableb,
                 int64_t e_lo, int64_t n_ent, const int64_t* lab_off, const int64_t* lab_col, int64_t nnz,
                 const int32_t* lab_perm, const float* tscale, float ls_add, float offset, const float* lse,
                 float inv_batch, const float* row_scale, float* dQ, float* dTable, float* rowstat_out, int flags,
                 void* ws, int64_t ws_bytes, cudaStream_t st, const TableUpdate* upd) {
  using namespace tcb;
  if (upd) {
    KGEB_REQUIRE(!dQ && !dTable && nnz == 0, "fused_bwd_update: dense table part only (label rows go through kgeb_fused_label_rows_to)");
    KGEB_REQUIRE(use_v2(), "fused_bwd_update: needs the v2 tile kernel (KGEB_BWD_V2=0 is set)");
    KGEB_REQUIRE(upd->w && upd->state && upd->mirror && upd->slot_of && upd->gbuf, "fused_bwd_update: NULL buffer");
    KGEB_REQUIRE(upd->mirror == tableb, "fused_bwd_update: the mirror to update must be the tile operand");
  }
  // KGEB_BWD_OVERWRITE_TABLE: the dense part is stored into dTable (no cleared buffer needed, no RMW); the label rows
  // are then scattered in AFTER the tile kernel instead of before it
  const bool overwrite = dTable && (flags & KGEB_BWD_OVERWRITE_TABLE);
  KGEB_REQUIRE(tc_bwd_supported(KGEB_MATH_BF16, d), "fused_bwd(bf16): entity dim must be a multiple of 16 and <= 256 (got %d)", d);
  KGEB_REQUIRE(Qb && tableb, "fused_bwd(bf16): the bf16 mirrors of Q and of the table are required");
  KGEB_REQUIRE(((reinterpret_cast<uintptr_t>(Qb) | reinterpret_cast<uintptr_t>(tableb)) & 15) == 0,
               "tensor tiles need 16-byte aligned operands");
  KGEB_REQUIRE(ws_bytes >= tc_bwd_workspace_bytes(B, d, n_ent, nnz), "fused_bwd(bf16): workspace too small");
  const int64_t nz = nnz < 1 ? 1 : nnz;
  char* wp = reinterpret_cast<char*>(ws);
  float* partial = reinterpret_cast<float*>(wp);      wp += a256((int64_t)kNumSMs * B * d * 4);
  float* dq_lab = reinterpret_cast<float*>(wp);       wp += a256(B * (int64_t)d * 4);
  float* rows_dq = reinterpret_cast<float*>(wp);      wp += a256(nz * (int64_t)d * 4);
  float* rows_dt = reinterpret_cast<float*>(wp);      wp += a256(nz * (int64_t)d * 4);
  int64_t* lab_ent = reinterpret_cast<int64_t*>(wp);  wp += a256(nz * 8);
  int64_t* lab_row = reinterpret_cast<int64_t*>(wp);  wp += a256(nz * 8);
  float* stat_partial = reinterpret_cast<float*>(wp); wp += a256((int64_t)kNumSMs * 4 * B * 2 * 4);
  float* entry_dot = reinterpret_cast<float*>(wp);    wp += a256(nz * 4);
  float* label_dot = reinterpret_cast<float*>(wp);    wp += a256(B * 4);
  const bool want_stats = rowstat_out != nullptr && dQ != nullptr && loss == KGEB_LOSS_BCE;
  void* scatter_ws = wp;
  const int64_t scatter_bytes = ws_bytes - (wp - reinterpret_cast<char*>(ws));
  int rc;
  CUtensorMap m_res, m_str;
  if (n_ent > 0 && B > 0) {
    // ---- sparse label part, forked onto the side stream --------------------------------------------------
    SideStream* ss = nullptr;
    if (nnz > 0) {
      ss = side_stream(dQ ? 0 : 1);
      KGEB_REQUIRE(ss, "fused_bwd(bf16): cannot create the side stream");
      cudaError_t e = cudaEventRecord(ss->fork, st);
      if (e == cudaSuccess) e = cudaStreamWaitEvent(ss->stream, ss->fork, 0);
      if (e != cudaSuccess) return cuda_status(e, "fused_bwd fork");
      cudaStream_t sd = ss->stream;
      label_entry_rows_kernel<<<(unsigned)((nnz + 8 * LABEL_EPW - 1) / (8 * LABEL_EPW)), 256, 0, sd>>>(
          Q, table, B, d, e_lo, n_ent, lab_off, lab_col, tscale, row_scale, inv_batch, nnz, dQ ? rows_dq : nullptr,
          dTable ? rows_dt : nullptr, lab_ent, lab_row, want_stats ? entry_dot : nullptr, offset);
      KGEB_LAUNCH_CHECK("label_entry_rows");
      if (dTable && !overwrite) {
        // label rows into the dense gradient before the tile kernel adds on top (it owns its rows; the order is fixed)
        rc = lab_perm ? kgeb_scatter_add_rows_perm(lab_ent, 1, lab_perm, rows_dt, nnz, d, dTable, n_ent, scatter_ws,
                                                   scatter_bytes, sd)
                      : kgeb_scatter_add_rows(lab_ent, 1, rows_dt, nnz, d, dTable, n_ent, scatter_ws, scatter_bytes, sd);
        if (rc) return rc;
      }
      if (dQ) {
        // label rows summed per query row (entries are grouped by row already) into a zeroed buffer that the partial
        // reduce adds in: the whole label part runs underneath the tile kernel
        e = cudaMemsetAsync(dq_lab, 0, (size_t)B * d * 4, sd);
        if (e != cudaSuccess) return cuda_status(e, "fused_bwd memset");
        if ((rc = scatter_add_rows_presorted(lab_row, rows_dq, nnz, d, dq_lab, B, scatter_ws, scatter_bytes, sd))) return rc;
      }
      if (want_stats) label_row_sum2_kernel<<<(unsigned)((B + 7) / 8), 256, 0, sd>>>(entry_dot, lab_off, B, label_dot);
      e = cudaEventRecord(ss->join, sd);
      if (e != cudaSuccess) return cuda_status(e, "fused_bwd join");
    }
    bool joined = (ss == nullptr);
    if (dQ) {
      Plan pl = make_plan(true, true, B, d, n_ent);
      if (pl.p.nstr < 2) { set_error("fused_bwd(bf16): not enough shared memory for dim %d", d); return KGEB_ERR_UNSUPPORTED; }
      pl.p.loss = loss; pl.p.offset = offset; pl.p.ls_add = ls_add; pl.p.inv_batch = inv_batch;
      pl.p.lse = lse; pl.p.row_scale = row_scale; pl.p.out = partial;
      pl.p.stat_partial = want_stats ? stat_partial : nullptr;
      if ((rc = make_map(&m_res, Qb, B, d, RES_ROWS, true)) || (rc = make_map(&m_str, tableb, n_ent, d, STR_ROWS, true))) return rc;
      const int64_t jobs = pl.p.n_res_blocks * pl.p.chunks;
      if ((rc = launch_bwd<true>(pl, m_res, m_str, m_res, jobs, st))) return rc;
      if (SideStream* s0 = side_stream(0)) cudaEventRecord(s0->tiles, st);   // the SMs are free again from here on
      if (!joined) {
        cudaError_t e = cudaStreamWaitEvent(st, ss->join, 0);
        if (e != cudaSuccess) return cuda_status(e, "fused_bwd join wait");
        joined = true;
      }
      const int64_t numel = B * (int64_t)d;
      const int64_t rblocks = (numel / 4 + 255) / 256;
      reduce_dq_partials_kernel<<<(unsigned)(rblocks > 4096 ? 4096 : rblocks), 256, 0, st>>>(
          partial, pl.p.chunks, numel, nnz > 0 ? dq_lab : nullptr, dQ);
      KGEB_LAUNCH_CHECK("reduce_dq_partials");
      if (want_stats) {   // BCE forward statistics came out of the same pass
        if (nnz == 0) cudaMemsetAsync(label_dot, 0, (size_t)B * 4, st);
        reduce_stat_partials_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(stat_partial, pl.p.chunks, B, label_dot,
                                                                                rowstat_out);
        KGEB_LAUNCH_CHECK("reduce_stat_partials");
      }
    }
    if (!joined) {
      cudaError_t e = cudaStreamWaitEvent(st, ss->join, 0);
      if (e != cudaSuccess) return cuda_status(e, "fused_bwd join wait");
    }
    if (dTable || upd) {
      Plan pl = make_plan(false, true, B, d, n_ent);
      if (pl.p.nstr < 2) { set_error("fused_bwd(bf16): not enough shared memory for dim %d", d); return KGEB_ERR_UNSUPPORTED; }
      pl.p.loss = loss; pl.p.offset = offset; pl.p.ls_add = ls_add; pl.p.inv_batch = inv_batch;
      pl.p.lse = lse; pl.p.row_scale = row_scale; pl.p.out = dTable;
      pl.p.overwrite = overwrite ? 1 : 0;
      if (upd) {
        pl.p.upd_w = upd->w; pl.p.upd_state = upd->state; pl.p.upd_mirror = reinterpret_cast<__nv_bfloat16*>(upd->mirror);
        pl.p.upd_slot = upd->slot_of; pl.p.upd_gbuf = upd->gbuf; pl.p.upd_skip = upd->skip;
        pl.p.upd_clr = upd->clr; pl.p.upd_eps = upd->eps; pl.p.upd_clr_dev = upd->clr_dev;
        pl.p.upd_debug = getenv("KGEB_UPD_DEBUG") ? atoi(getenv("KGEB_UPD_DEBUG")) : 0;
        // tuning knob, off by default: spread the CTAs' phases over one job period (KGEB_UPD_STAGGER = clocks per tile, e.g.
        // 1100).  Measured with 0 / 1100 / 2200: no difference -- the CTAs do not run in lockstep -- and the last CTA's
        // start delay of one job period is 3 % of the kernel on an eighth of the table.
        static const int stagger_tile_clk = getenv("KGEB_UPD_STAGGER") ? atoi(getenv("KGEB_UPD_STAGGER")) : 0;
        const int64_t grid = pl.p.n_res_blocks < kNumSMs ? pl.p.n_res_blocks : kNumSMs;
        pl.p.stagger_clk = pl.p.n_res_blocks > 2 * grid ? (int)(pl.p.n_str_tiles * stagger_tile_clk / grid) : 0;
      }
      if (loss == KGEB_LOSS_KL && pl.p.colk_n > 0) {
        // (label_dot's slot of the workspace is free in a dTable-only call; with dQ in the same call it is used by the
        // BCE statistics only, never by KL)
        float* colk = reinterpret_cast<float*>(dq_lab);     // [B * d] floats: room for colk_n <= 4096 + 63
        colk_kernel<<<(pl.p.colk_n + 255) / 256, 256, 0, st>>>(lse, row_scale, inv_batch, B, pl.p.colk_n, colk);
        KGEB_LAUNCH_CHECK("colk");
        pl.p.colk = colk;
      } else {
        pl.p.colk_n = 0;
      }
      CUtensorMap m_out;   // fp32 [n_ent, d], boxes of 32 columns x 128 rows for the reduce-add flush
      if ((rc = make_map(&m_res, tableb, n_ent, d, RES_ROWS, true)) || (rc = make_map(&m_str, Qb, B, d, STR_ROWS, true)) ||
          (rc = make_map(&m_out, upd ? upd->w : dTable, n_ent, d, RES_ROWS, false)))     // (unused by the fused update)
        return rc;
      const int64_t jobs = pl.p.n_res_blocks;
      if ((rc = launch_bwd<false>(pl, m_res, m_str, m_out, jobs, st))) return rc;
      if (overwrite && nnz > 0) {   // label rows on top of the stored dense part (joined with the side stream above)
        rc = lab_perm ? kgeb_scatter_add_rows_perm(lab_ent, 1, lab_perm, rows_dt, nnz, d, dTable, n_ent, scatter_ws,
                                                   scatter_bytes, st)
                      : kgeb_scatter_add_rows(lab_ent, 1, rows_dt, nnz, d, dTable, n_ent, scatter_ws, scatter_bytes, st);
        if (rc) return rc;
      }
    }
  } else {
    if (dQ && B > 0) cudaMemsetAsync(dQ, 0, (size_t)B * d * 4, st);
    if (overwrite && n_ent > 0) cudaMemsetAsync(dTable, 0, (size_t)n_ent * d * 4, st);
  }
  return KGEB_OK;
}

// FLASH forward (KL, bf16 tiles): row statistics and o_sum = sum_e exp(x - mref) * table[e] in one pass over the table.
int tc_flash_fwd(const float* Q, const void* Qb, int64_t B, int d, const float* table, const void* tableb, int64_t e_lo,
                 int64_t n_ent, const int64_t* lab_off, const int64_t* lab_col, int64_t nnz, float* rowstat, float* o_sum,
                 int* status, void* ws, int64_t ws_bytes, cudaStream_t st) {
  using namespace tcb;
  KGEB_REQUIRE(tc_bwd_supported(KGEB_MATH_BF16, d), "fused_flash_fwd: entity dim must be a multiple of 16 and <= 256 (got %d)", d);
  KGEB_REQUIRE(Qb && tableb, "fused_flash_fwd: the bf16 mirrors of Q and of the table are required");
  KGEB_REQUIRE(ws_bytes >= tc_bwd_workspace_bytes(B, d, n_ent, nnz), "fused_flash_fwd: workspace too small");
  const int64_t nz = nnz < 1 ? 1 : nnz;
  char* wp = reinterpret_cast<char*>(ws);
  float* partial = reinterpret_cast<float*>(wp);      wp += a256((int64_t)kNumSMs * B * d * 4);
  wp += a256(B * (int64_t)d * 4) + 2 * a256(nz * (int64_t)d * 4);
  int64_t* lab_ent = reinterpret_cast<int64_t*>(wp);  wp += a256(nz * 8);
  int64_t* lab_row = reinterpret_cast<int64_t*>(wp);  wp += a256(nz * 8);
  float* stat_partial = reinterpret_cast<float*>(wp); wp += a256((int64_t)kNumSMs * 4 * B * 2 * 4);
  float* entry_dot = reinterpret_cast<float*>(wp);    wp += a256(nz * 4);
  float* label_dot = reinterpret_cast<float*>(wp);    wp += a256(B * 4);
  float* mref = reinterpret_cast<float*>(wp);         wp += a256(B * 4);
  if (B == 0) return KGEB_OK;
  // exact fp32 scores at the label entries of this shard (their sum per row enters the loss value)
  if (nnz > 0) {
    label_entry_rows_kernel<<<(unsigned)((nnz + 8 * LABEL_EPW - 1) / (8 * LABEL_EPW)), 256, 0, st>>>(
        Q, table, B, d, e_lo, n_ent, lab_off, lab_col, nullptr, nullptr, 1.f, nnz, nullptr, nullptr, lab_ent, lab_row,
        entry_dot, 0.f);
    KGEB_LAUNCH_CHECK("label_entry_rows");
    label_row_sum2_kernel<<<(unsigned)((B + 7) / 8), 256, 0, st>>>(entry_dot, lab_off, B, label_dot);
  } else {
    cudaMemsetAsync(label_dot, 0, (size_t)B * 4, st);
  }
  if (n_ent <= 0) {   // an empty shard contributes nothing: (max, sum) = (-inf, 0)
    cudaMemsetAsync(o_sum, 0, (size_t)B * d * 4, st);
    flash_rowstat_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(nullptr, 0, B, nullptr, label_dot, rowstat);
    KGEB_LAUNCH_CHECK("flash_rowstat");
    return KGEB_OK;
  }
  sample_max_kernel<<<(unsigned)((B + kFlashRows - 1) / kFlashRows), kFlashWarps * 32, 0, st>>>(
      Q, table, B, d, e_lo, n_ent, lab_off, lab_col, nnz > 0 ? entry_dot : nullptr, mref);
  KGEB_LAUNCH_CHECK("sample_max");
  Plan pl = make_plan(true, true, B, d, n_ent);
  if (pl.p.nstr < 2) { set_error("fused_flash_fwd: not enough shared memory for dim %d", d); return KGEB_ERR_UNSUPPORTED; }
  pl.p.loss = KGEB_LOSS_KL; pl.p.inv_batch = 1.f; pl.p.out = partial; pl.p.stat_partial = stat_partial; pl.p.mref = mref;
  pl.p.status = status;
  CUtensorMap m_res, m_str;
  int rc;
  if ((rc = make_map(&m_res, Qb, B, d, RES_ROWS, true)) || (rc = make_map(&m_str, tableb, n_ent, d, STR_ROWS, true))) return rc;
  if ((rc = launch_bwd<true>(pl, m_res, m_str, m_res, pl.p.n_res_blocks * pl.p.chunks, st, true))) return rc;
  if (SideStream* s0 = side_stream(0)) cudaEventRecord(s0->tiles, st);
  const int64_t numel = B * (int64_t)d;
  const int64_t rblocks = (numel / 4 + 255) / 256;
  reduce_dq_partials_kernel<<<(unsigned)(rblocks > 4096 ? 4096 : rblocks), 256, 0, st>>>(partial, pl.p.chunks, numel, nullptr, o_sum);
  KGEB_LAUNCH_CHECK("reduce_dq_partials");
  flash_rowstat_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(stat_partial, pl.p.chunks, B, mref, label_dot, rowstat);
  KGEB_LAUNCH_CHECK("flash_rowstat");
  return KGEB_OK;
}

// FLASH backward for the queries: no table pass -- o_sum is rescaled by the (global) log-sum-exp and the exact fp32 label
// rows are added.
int tc_flash_dq(const float* Q, int64_t B, int d, const float* table, int64_t e_lo, int64_t n_ent, const int64_t* lab_off,
                const int64_t* lab_col, int64_t nnz, const float* tscale, const float* rowstat_local, const float* lse,
                float inv_batch, const float* row_scale, const float* o_sum, float* dQ, void* ws, int64_t ws_bytes,
                cudaStream_t st) {
  using namespace tcb;
  KGEB_REQUIRE(ws_bytes >= tc_bwd_workspace_bytes(B, d, n_ent, nnz), "fused_flash_dq: workspace too small");
  if (B == 0) return KGEB_OK;
  const int64_t nz = nnz < 1 ? 1 : nnz;
  char* wp = reinterpret_cast<char*>(ws);
  wp += a256((int64_t)kNumSMs * B * d * 4);
  float* dq_lab = reinterpret_cast<float*>(wp);       wp += a256(B * (int64_t)d * 4);
  float* rows_dq = reinterpret_cast<float*>(wp);      wp += 2 * a256(nz * (int64_t)d * 4);
  int64_t* lab_ent = reinterpret_cast<int64_t*>(wp);  wp += a256(nz * 8);
  int64_t* lab_row = reinterpret_cast<int64_t*>(wp);  wp += a256(nz * 8);
  wp += a256((int64_t)kNumSMs * 4 * B * 2 * 4) + a256(nz * 4) + 2 * a256(B * 4);
  void* scatter_ws = wp;
  const int64_t scatter_bytes = ws_bytes - (wp - reinterpret_cast<char*>(ws));
  int rc;
  const bool labels = nnz > 0 && n_ent > 0;
  if (labels) {
    label_entry_rows_kernel<<<(unsigned)((nnz + 8 * LABEL_EPW - 1) / (8 * LABEL_EPW)), 256, 0, st>>>(
        Q, table, B, d, e_lo, n_ent, lab_off, lab_col, tscale, row_scale, inv_batch, nnz, rows_dq, nullptr, lab_ent, lab_row,
        nullptr, 0.f);
    KGEB_LAUNCH_CHECK("label_entry_rows");
    cudaError_t e = cudaMemsetAsync(dq_lab, 0, (size_t)B * d * 4, st);
    if (e != cudaSuccess) return cuda_status(e, "fused_flash_dq memset");
    if ((rc = scatter_add_rows_presorted(lab_row, rows_dq, nnz, d, dq_lab, B, scatter_ws, scatter_bytes, st))) return rc;
  }
  const int64_t rblocks = (B * (int64_t)d / 4 + 255) / 256;
  flash_dq_kernel<<<(unsigned)(rblocks > 4096 ? 4096 : rblocks), 256, 0, st>>>(o_sum, rowstat_local, lse, lab_off, inv_batch,
                                                                              row_scale, labels ? dq_lab : nullptr, B, d, dQ);
  KGEB_LAUNCH_CHECK("flash_dq");
  return KGEB_OK;
}

// The sparse label part of the dense table gradient on its own (kgeb_fused_label_rows): lets a caller route the label
// rows into a different buffer than the tile kernel's output, so that the tile kernel does not have to wait for them.
int tc_label_rows(const float* Q, int64_t B, int d, const float* table, int64_t e_lo, int64_t n_ent, const int64_t* lab_off,
                  const int64_t* lab_col, int64_t nnz, const int32_t* lab_perm, const float* tscale, const float* row_scale,
                  float inv_batch, float* dense_out, void* ws, int64_t ws_bytes, cudaStream_t st, const int64_t* out_rows,
                  int64_t n_out) {
  using namespace tcb;
  if (nnz <= 0 || n_ent <= 0 || B <= 0) return KGEB_OK;
  char* wp = reinterpret_cast<char*>(ws);
  float* rows_dt = reinterpret_cast<float*>(wp);      wp += a256(nnz * (int64_t)d * 4);
  int64_t* lab_ent = reinterpret_cast<int64_t*>(wp);  wp += a256(nnz * 8);
  int64_t* lab_row = reinterpret_cast<int64_t*>(wp);  wp += a256(nnz * 8);
  const int64_t scatter_bytes = ws_bytes - (wp - reinterpret_cast<char*>(ws));
  KGEB_REQUIRE(scatter_bytes >= kgeb_scatter_workspace_bytes(nnz, d), "fused_label_rows: workspace too small");
  label_entry_rows_kernel<<<(unsigned)((nnz + 8 * LABEL_EPW - 1) / (8 * LABEL_EPW)), 256, 0, st>>>(
      Q, table, B, d, e_lo, n_ent, lab_off, lab_col, tscale, row_scale, inv_batch, nnz, nullptr, rows_dt, lab_ent, lab_row,
      nullptr, 0.f);
  KGEB_LAUNCH_CHECK("label_entry_rows");
  // out_rows: the rows go to dense_out[out_rows[i]] ([n_out, d]) instead of dense_out[entity - e_lo]; entries of other
  // shards carry zero rows either way.  lab_perm must then sort out_rows as well (equal keys contiguous).
  const int64_t* keys = out_rows ? out_rows : lab_ent;
  const int64_t vocab = out_rows ? n_out : n_ent;
  return lab_perm ? kgeb_scatter_add_rows_perm(keys, 1, lab_perm, rows_dt, nnz, d, dense_out, vocab, wp, scatter_bytes, st)
                  : kgeb_scatter_add_rows(keys, 1, rows_dt, nnz, d, dense_out, vocab, wp, scatter_bytes, st);
}

int tc_wait_tiles(cudaStream_t st) {
  SideStream* s0 = side_stream(0);
  KGEB_REQUIRE(s0, "fused_bwd_wait_tiles: cannot create the event");
  cudaError_t e = cudaStreamWaitEvent(st, s0->tiles, 0);
  if (e != cudaSuccess) return cuda_status(e, "fused_bwd_wait_tiles");
  return KGEB_OK;
}

}  // namespace kgeb

#ifdef KGEB_TRACE
// tuning builds: copies the trace of block 0 to the host and resets it; returns the number of events
extern "C" int kgeb_debug_trace(unsigned long long* host_dst, int max_n) {
  // all 32 x 2048 slots (zero = unused); cleared for the next launch
  const int n = 32 << 11;
  if (max_n < n) return -1;
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(host_dst, kgeb::tcb::g_trace, sizeof(unsigned long long) * n);
  void* p = nullptr;
  cudaGetSymbolAddress(&p, kgeb::tcb::g_trace);
  cudaMemset(p, 0, sizeof(unsigned long long) * n);
  return n;
}
#endif
