/* kgeb200 -- C-ABI of the B200-native (sm_100a) LibKGE scoring/embedding hot path.
 *
 * Every entry point takes plain device pointers, sizes and a CUDA stream (void* = cudaStream_t;
 * NULL = legacy default stream) and returns an int status (KGEB_OK / KGEB_ERR_*); the text of the
 * last failure on the calling thread is returned by kgeb_last_error().  No torch types appear in
 * any signature.  All matrices are row-major, contiguous fp32; index arrays are int32 or int64
 * (flag idx64), matching the reference (int64 in training, train.py:622,811,1022; int32 in
 * evaluation, dataset.py:178 / entity_ranking.py:76).  A NULL index pointer means "row i".
 *
 * Each function cites the reference interface (file:line under Nzteb/kge-1) it replaces.
 * The reference is pure Python/PyTorch, so the binding a maintainer adds is a ctypes stub; it is
 * shown in INTEGRATION.md and implemented in kge-1_b200/lib.py.
 */
#ifndef KGEB200_H
#define KGEB200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KGEB_OK 0
#define KGEB_ERR_ARG 1         /* bad argument -> ValueError in the binding */
#define KGEB_ERR_CUDA 2        /* CUDA runtime / driver error -> RuntimeError */
#define KGEB_ERR_UNSUPPORTED 3 /* valid in the reference, not built here -> NotImplementedError */

/* kge/model/{distmult,complex,cp,simple,rescal,transe,rotate}.py */
enum { KGEB_DISTMULT = 0, KGEB_COMPLEX = 1, KGEB_CP = 2, KGEB_SIMPLE = 3, KGEB_RESCAL = 4,
       KGEB_TRANSE = 5, KGEB_ROTATE = 6 };
/* combine= of RelationalScorer.score_emb (kge_model.py:120-182) */
enum { KGEB_SP_ = 0, KGEB__PO = 1 };
/* score of one (query vector q, candidate row c) pair -- SURVEY.md Appendix D:
 *   DOT    sum_k q_k c_k                 (DistMult, ComplEx, CP, SimplE, RESCAL)
 *   NEG_L1 -sum_k |q_k - c_k|            (TransE l_norm=1, transe.py:19-21)
 *   NEG_L2 -sqrt(sum_k (q_k - c_k)^2)    (TransE l_norm=2)
 *   ROT_L1 +sum_{k<d/2} |q_k - c_k|_C    (RotatE l_norm=1, rotate.py:41-60; positive distance)
 *   ROT_L2 +sqrt(sum_{k<d/2} |q_k - c_k|_C^2)                                              */
enum { KGEB_DOT = 0, KGEB_NEG_L1 = 1, KGEB_NEG_L2 = 2, KGEB_ROT_L1 = 3, KGEB_ROT_L2 = 4 };
/* kge/util/loss.py: KLDivWithSoftmaxKgeLoss (192-213), BCEWithLogitsKgeLoss bce_type=None (137-159) */
enum { KGEB_LOSS_KL = 0, KGEB_LOSS_BCE = 1 };
/* arithmetic of the all-entity DOT tiles */
enum { KGEB_MATH_FP32 = 0,   /* CUDA-core FFMA, fp32 (1e-5 bar)                                         */
       KGEB_MATH_TF32 = 1,   /* tcgen05.mma kind::tf32 on the fp32 tables in place, fp32 accumulate in TMEM */
       KGEB_MATH_BF16 = 2 }; /* tcgen05.mma kind::f16 on bf16 mirrors (kgeb_to_bf16), fp32 accumulate      */

const char* kgeb_last_error(void);
/* library build info: returns the compiled arch (100) and writes a version string */
int kgeb_version(char* buf, int buflen);

/* ---- a1/K1: LookupEmbedder.embed (embedder/lookup_embedder.py:91-92): out[i,:] = W[idx[i],:] ---- */
int kgeb_gather_rows(const float* W, int64_t vocab, int dim, const void* idx, int idx64, int64_t n,
                     float* out, void* stream);

/* Entity-sharded tables (SURVEY.md 8e): W_shard holds the rows [e_lo, e_hi) of the global table.  out[i,:] = the row of
 * idx[i] if this shard owns it, zeros otherwise (an all-reduce over the shards assembles the rows); local_ids[i]
 * (optional) = idx[i] - e_lo, or e_hi - e_lo ("not mine": the dummy row a sharded scatter adds such gradients to). */
int kgeb_gather_rows_shard(const float* W_shard, int64_t e_lo, int64_t e_hi, int dim, const void* idx, int idx64,
                           int64_t n, float* out, int64_t* local_ids, void* stream);

/* ---- a4/K5: score_emb(..., "spo") for the seven scorers, fused with the three gathers.
 * x_src point at [vocab,d] tables (with x_idx) or at [n,d] embedding matrices (x_idx NULL).
 * p rows have relation_dim(model,d) columns (d, d/2 for CP/RotatE, d*d for RESCAL).
 * l_norm in {1,2} (TransE/RotatE).  TransE adds eps=1e-6 to the difference (pairwise_distance). */
int kgeb_score_spo(int model, int l_norm, const float* s_src, const void* s_idx, const float* p_src,
                   const void* p_idx, const float* o_src, const void* o_idx, int idx64, int64_t n, int d,
                   float* out, void* stream);
/* autograd of the above (reference: ATen backward of the expressions in <model>.py); writes per-row
 * gradients ds[n,d], dp[n,dr], do[n,d] (not accumulated; scatter them with kgeb_scatter_add_rows). */
int kgeb_score_spo_bwd(int model, int l_norm, const float* s_src, const void* s_idx, const float* p_src,
                       const void* p_idx, const float* o_src, const void* o_idx, int idx64, int64_t n,
                       int d, const float* gout, float* ds, float* dp, float* d_o, void* stream);

/* ---- query transform of the sp_/_po forms (SURVEY.md App. D; <model>.py score_emb "sp_"/"_po"):
 * Q[i,:] = q(a_i, p_i), a = s for KGEB_SP_, a = o for KGEB__PO; Q is [n,d].  */
int kgeb_query_build(int model, int combine, const int32_t* row_combine /* per-row KGEB_SP_/KGEB__PO, or NULL */,
                     const float* a_src, const void* a_idx, const float* p_src, const void* p_idx, int idx64,
                     int64_t n, int d, float* Q, void* stream);
/* chain rule dQ -> da[n,d], dp[n,dr] */
int kgeb_query_bwd(int model, int combine, const int32_t* row_combine, const float* a_src, const void* a_idx,
                   const float* p_src, const void* p_idx, int idx64, int64_t n, int d, const float* dQ, float* da,
                   float* dp, void* stream);

/* ---- negative-sampling pair scoring (train.py:872-893 "triple" implementation without the
 * B*(1+N) expansion): out[i,j] = pair_score(kind, Q[i,:], table[cand[i,j],:]), cand is [B,M]. */
int kgeb_pairs_score(int kind, const float* Q, const float* table, const void* cand, int idx64, int64_t B,
                     int64_t M, int d, float* out, void* stream);
/* backward: G[B,M] = dL/dout -> dQ[B,d] and per-pair candidate gradients dC[B*M,d] */
int kgeb_pairs_bwd(int kind, const float* Q, const float* table, const void* cand, int idx64, int64_t B,
                   int64_t M, int d, const float* G, const float* scores, float* dQ, float* dC, void* stream);

/* negative-sampling batch body without autograd (train.py:853-994, implementation "triple"):
 * candidates [B,1+N] = (positive target | negatives); loss over the score rows with label column 0
 * (KL = cross entropy, loss.py:195-208; BCE with offset, loss.py:153-159): writes G = dL/dscores [B,1+N] and
 * the per-row loss, both already divided by the batch size (inv_batch). */
int kgeb_ns_candidates(const int64_t* target, const int64_t* negatives, int64_t B, int64_t N, int64_t* cand,
                       void* stream);
int kgeb_ns_loss(int loss, const float* scores, int64_t B, int64_t M, float offset, float inv_batch, float* G,
                 float* row_loss, void* stream);

/* ---- a5/a6/K4/K6/K7: score_emb(..., "sp_"|"_po") materialised:
 * out[i*ld + col_off + j] = pair_score(kind, Q[i,:], table[cand_idx ? cand_idx[j] : j, :]), j < m.
 * math = KGEB_MATH_FP32 | KGEB_MATH_TF32 (TF32 only for KGEB_DOT). */
int kgeb_score_all(int kind, int math, const float* Q, int64_t B, int d, const float* table,
                   const void* cand_idx, int idx64, int64_t m, float* out, int64_t ld, int64_t col_off,
                   void* stream);
/* backward of the materialised form: G is [B, ld] (columns col_off..col_off+m used), X the forward
 * scores (needed by the L2 kinds).  dQ[B,d] is overwritten, dC[m,d] overwritten (row j = candidate j). */
int kgeb_score_all_bwd(int kind, const float* Q, int64_t B, int d, const float* table, const void* cand_idx,
                       int idx64, int64_t m, const float* G, const float* X, int64_t ld, int64_t col_off,
                       float* dQ, float* dC, void* stream);

/* The sparse label part of kgeb_fused_bwd's dense table gradient on its own: for every label entry (row q, entity e)
 * dTable_out[e - e_lo, :] += -inv_batch * grad_scale[q] * t_q * Q[q, :]  (t_q as in kgeb_fused_bwd; fixed-order segment
 * sums, lab_perm as there).  A caller that sends these rows to a second gradient buffer and calls kgeb_fused_bwd with
 * nnz = 0 for the dense part removes the label chain from the tile kernel's critical path (the optimizer adds the two
 * buffers anyway, kgeb_adagrad_dense grad / grad2).  Workspace: kgeb_fused_workspace_bytes(B, d, e_hi - e_lo, nnz). */
/* Makes `stream` wait for the dQ tile kernel of the calling thread's most recent kgeb_fused_bwd(dQ != NULL, bf16 tiles)
 * on this device -- not for the small reduction kernels that follow it: a second persistent tile kernel (the dense
 * dTable half) queued on `stream` starts the moment the first one releases the SMs.  Event wait: capturable. */
int kgeb_fused_bwd_wait_tiles(void* stream);
int kgeb_fused_label_rows(int loss, const float* Q, int64_t B, int d, const float* table, int64_t e_lo, int64_t e_hi,
                          const int64_t* lab_off, const int64_t* lab_col, int64_t nnz, const int32_t* lab_perm,
                          float label_smoothing, float inv_batch, const float* grad_scale, float* dTable_out,
                          void* workspace, int64_t workspace_bytes, void* stream);

/* kgeb_fused_label_rows with entry i routed to dense_out[out_rows[i]] ([n_out, d]) instead of dense_out[entity - e_lo]
 * (lab_perm, when given, must keep equal out_rows values contiguous: true for slots numbered in entity order). */
int kgeb_fused_label_rows_to(int loss, const float* Q, int64_t B, int d, const float* table, int64_t e_lo, int64_t e_hi,
                             const int64_t* lab_off, const int64_t* lab_col, int64_t nnz, const int32_t* lab_perm,
                             float label_smoothing, float inv_batch, const float* grad_scale, const int64_t* out_rows,
                             int64_t n_out, float* dense_out, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- optimizer.step() inside the table-gradient kernel (train.py:323 backward + :375 optimizer.step for the entity table).
 * For an [E, d] table the dense gradient G^T Q is as large as the table; storing it and reading it back in an Adagrad pass
 * costs 2 x E*d*4 bytes of HBM traffic per step.  A CTA of the tile kernel that has finished an entity tile holds the
 * complete dense gradient of its 128 rows in tensor memory and applies Adagrad from there.  Rows that also receive sparse
 * gradient rows in this step (label rows, query-side rows: <= 8192 ids) are excluded and handled by a row kernel:
 *   kgeb_touched_build   sorts the ids (ids_a ++ ids_b, global entity ids; those outside [e_lo, e_hi) are ignored), numbers
 *                        the distinct ones 0..n-1 in ascending order: slot_of[id - e_lo] = slot (the caller keeps slot_of
 *                        [e_hi - e_lo] at -1 between steps), uniq_rows[slot] = id - e_lo, *num_uniq = n, and
 *                        slot_a[i] / slot_b[i] = slot of position i (n_a + n_b = the dummy slot for ids of other shards);
 *   kgeb_fused_bwd_update  the dense part (bf16 tiles, KGEB_LOSS_*; arguments as kgeb_fused_bwd): slot_of[row] < 0 ->
 *                        Adagrad on W / state / bf16 mirror in the flush; else the row goes to gbuf[slot];
 *   (the caller scatters its sparse rows into g_sparse [n_a + n_b + 1, d] by slot: kgeb_fused_label_rows_to,
 *    kgeb_scatter_add_rows[_perm] with slot_a as the index)
 *   kgeb_touched_update  Adagrad on the touched rows with gbuf[slot] + g_sparse[slot]; clears g_sparse and slot_of again.
 * skip_flag (optional device word): non-zero = neither kernel changes W, the state or the mirror (failed flash pass).
 * The arithmetic is kgeb_adagrad_dense's, operation for operation (weight_decay = 0). */
int kgeb_touched_capacity(void);
int kgeb_touched_build(const int64_t* ids_a, int64_t n_a, const int64_t* ids_b, int64_t n_b,
                       const int64_t* n_b_real /* device: ids_b past this count are padding (slot 0, not touched); or NULL */,
                       int64_t e_lo, int64_t e_hi, int32_t* slot_of, int64_t* uniq_rows, int64_t* num_uniq, int64_t* slot_a,
                       int64_t* slot_b, void* stream);
int kgeb_fused_bwd_update(int loss, const float* Q, int64_t B, int d, float* table, int64_t e_lo, int64_t e_hi,
                          int64_t num_entities, const int64_t* lab_off, float label_smoothing, float offset,
                          const float* lse, float inv_batch, const float* grad_scale, void* table_bf16, float* state,
                          float clr, float eps, const int32_t* slot_of, float* gbuf, const int32_t* skip_flag,
                          void* workspace, int64_t workspace_bytes, void* stream);
int kgeb_touched_update(float* W, float* state, void* bf16_mirror, int32_t* slot_of, const int64_t* uniq_rows,
                        const int64_t* num_uniq, int64_t capacity /* n_a + n_b */, const float* g_dense, float* g_sparse,
                        int d, float clr, float eps, const int32_t* skip_flag, void* stream);
/* _sched siblings: the effective learning rate clr = lr / (1 + (step - 1) * lr_decay) of the step is read from the device
 * word *clr (non-NULL) instead of being passed by value, so that a captured CUDA graph follows a learning-rate schedule
 * when the caller rewrites the word between replays.  Same kernels as the by-value entries (the word is read once per
 * thread): a given rate gives the same bits either way. */
int kgeb_fused_bwd_update_sched(int loss, const float* Q, int64_t B, int d, float* table, int64_t e_lo, int64_t e_hi,
                                int64_t num_entities, const int64_t* lab_off, float label_smoothing, float offset,
                                const float* lse, float inv_batch, const float* grad_scale, void* table_bf16, float* state,
                                const float* clr, float eps, const int32_t* slot_of, float* gbuf, const int32_t* skip_flag,
                                void* workspace, int64_t workspace_bytes, void* stream);
int kgeb_touched_update_sched(float* W, float* state, void* bf16_mirror, int32_t* slot_of, const int64_t* uniq_rows,
                              const int64_t* num_uniq, int64_t capacity, const float* g_dense, float* g_sparse, int d,
                              const float* clr, float eps, const int32_t* skip_flag, void* stream);

/* ---- K4+K8+K9 fused all-entity training (DOT kinds): scores are never materialised.
 * Labels are a CSR over the batch rows: lab_off[B+1] (int64), lab_col[nnz] (int64, ascending within a
 * row, entity ids).  For 1vsAll each row has exactly one label.  Targets t_ij:
 *   BCE: t = (1-ls)*y + ls_add           (train.py:715-721; ls_add = 1/E when ls>0 else 0)
 *   KL : t = normalize_L1((1-ls)*y + ls_add) (loss.py:211-213), index labels = one-hot
 * Entities [e_lo, e_hi) of `table` (row e of table = entity e_lo + e .. the table pointer is the shard's
 * first row) are scored; num_entities is the global E (for ls_add and KL normalisation).
 * fwd: per-row statistics of this shard, rowstat[i*4 + k]:
 *   k=0  KL : max_j x_ij                         BCE: sum_j softplus(x_ij + offset)
 *   k=1  KL : sum_j exp(x_ij - max)              BCE: unused
 *   k=2  sum_j (x_ij [+ offset for BCE])         (dense part of the target, label smoothing)
 *   k=3  sum over the row's label entries in this shard of (x_ij [+ offset for BCE])
 *   from which the caller forms the loss (kge-1_b200/fused.py) and, across shards, the global
 *   log-sum-exp.  KL with label_smoothing != 0 returns KGEB_ERR_UNSUPPORTED.
 * bwd: G_ij = inv_batch * (softmax_ij * tsum_i - t_ij)  (KL, lse[i] = global log-sum-exp)
 *      G_ij = inv_batch * (sigmoid(x_ij + offset) - t_ij) (BCE);
 *   dQ[B,d] = G * table (overwritten with this shard's partial), dTable[e,:] += G^T Q.      */
int kgeb_fused_fwd(int loss, int math, const float* Q, int64_t B, int d, const float* table, int64_t e_lo,
                   int64_t e_hi, int64_t num_entities, const int64_t* lab_off, const int64_t* lab_col,
                   int64_t nnz /* size of lab_col (>= lab_off[B]; the tail may be padding) */, float label_smoothing, float offset, const void* table_bf16 /* mirror, KGEB_MATH_BF16 only */,
                   float* rowstat /* kgeb_fused_bwd flags.  KGEB_BWD_OVERWRITE_TABLE: dTable[e_lo..e_hi) is OVERWRITTEN with the gradient (dense part stored by
 * the tile kernel with plain TMA stores, label rows scattered on top afterwards) instead of accumulated into: the caller
 * needs no cleared buffer and the L2 does no read-modify-write -- at the Wikidata5M shape that is 2 x 2.4 GB of HBM traffic
 * per step (embedding_dense_backward of the reference zero-fills and accumulates, K3). */
#define KGEB_BWD_OVERWRITE_TABLE 1
/*[B,4]*/, void* workspace, int64_t workspace_bytes, void* stream);
int kgeb_fused_bwd(int loss, int math, const float* Q, int64_t B, int d, const float* table, int64_t e_lo,
                   int64_t e_hi, int64_t num_entities, const int64_t* lab_off, const int64_t* lab_col,
                   int64_t nnz /* size of lab_col (>= lab_off[B]; the tail may be padding) */,
                   const int32_t* lab_perm /* [nnz] or NULL: stable argsort of lab_col[0..nnz) (entries grouped by
                                              entity, positions ascending), as the batch collate can provide it; spares
                                              the device sort of the label scatter into dTable (BF16 tiles) */,
                   float label_smoothing, float offset, const float* lse /*[B] (KL)*/, float inv_batch,
                   const float* row_scale /*[B] per-row factor multiplied into G (upstream gradient), or NULL*/,
                   const void* table_bf16 /* mirror, KGEB_MATH_BF16 only */, float* dQ, float* dTable,
                   float* rowstat_out /* [B,4] or NULL: also produce the forward statistics of kgeb_fused_fwd (BCE on the
                                         bf16 tiles gets them from the same pass; otherwise the forward kernels run) */,
                   int flags /* 0 | KGEB_BWD_OVERWRITE_TABLE */, void* workspace, int64_t workspace_bytes, void* stream);
/* kgeb_fused_fwd / kgeb_fused_bwd for every pair kind on the fp32 CUDA-core tiles: the fused score + loss of TransE
 * (KGEB_NEG_L1 / _L2, transe.py:14-24) and RotatE (KGEB_ROT_L1 / _L2, rotate.py:18-63, 97-145) under the KL and BCE
 * losses (loss.py:137-159, 192-213), without the [B, E] score matrix.  Same statistics layout, workspace
 * (kgeb_fused_workspace_bytes), label CSR, shard range, KGEB_BWD_OVERWRITE_TABLE and results as the two entries above;
 * scores are those of kgeb_score_all (RotatE +distance, TransE without eps) and gradients follow kgeb_score_all_bwd
 * (sign(0) = 0, zero distance or zero modulus -> zero gradient).  kind == KGEB_DOT is kgeb_fused_fwd / _bwd with
 * KGEB_MATH_FP32.  KGEB_ERR_UNSUPPORTED: d > 256, KL with label smoothing; an odd d for RotatE is an argument error. */
int kgeb_fused_fwd_kind(int kind, int loss, const float* Q, int64_t B, int d, const float* table, int64_t e_lo,
                        int64_t e_hi, int64_t num_entities, const int64_t* lab_off, const int64_t* lab_col, int64_t nnz,
                        float label_smoothing, float offset, float* rowstat /*[B,4]*/, void* workspace,
                        int64_t workspace_bytes, void* stream);
int kgeb_fused_bwd_kind(int kind, int loss, const float* Q, int64_t B, int d, const float* table, int64_t e_lo,
                        int64_t e_hi, int64_t num_entities, const int64_t* lab_off, const int64_t* lab_col, int64_t nnz,
                        float label_smoothing, float offset, const float* lse /*[B] (KL)*/, float inv_batch,
                        const float* row_scale /*[B] or NULL*/, float* dQ, float* dTable,
                        int flags /* 0 | KGEB_BWD_OVERWRITE_TABLE */, void* workspace, int64_t workspace_bytes,
                        void* stream);
/* loss(scores, labels) / batch_size from the (shard-combined) forward statistics, as the reference's loss objects
 * return it (loss.py:153-159, 198-213): rows_out[B] per-row values (may be NULL), lse_out[B] log-sum-exp per row for
 * the KL backward (may be NULL), total[1] their sum in a fixed order. */
int kgeb_loss_from_rowstat(int loss, const float* rowstat, const int64_t* lab_off, int64_t B, float label_smoothing,
                           int64_t num_entities, float inv_batch, float* rows_out, float* lse_out, float* total,
                           void* stream);
/* KL on the bf16 tiles with the forward statistics and the query gradient in ONE pass over the table (the forward kernel of
 * kgeb_fused_fwd and the score recomputation of the dQ half of kgeb_fused_bwd fall away: 4 instead of 5 GEMM passes and 2
 * instead of 3 exponentials per score and step).  Per score P = exp(x - mref_q) is computed once against a FIXED per-row
 * reference (mref_q = max of x over a strided sample of 64 entities of the shard, shifted by min(2 sigma, 40)); the row sums of P accumulate in
 * registers, o_sum[q,:] = sum_e P[q,e] * table[e,:] in tensor memory.  No online rescaling: bf16 operands and fp32
 * accumulators keep 8 exponent bits, so P is representable for x up to ~88 nats above mref (terms far below it underflow
 * harmlessly).  mref also covers the batch's label entities and the row's own labels -- where a trained model puts its
 * large scores.  It remains a guess: *status (device, int32; the caller zeroes it) is set to 1 when a row sum or an
 * accumulator left the fp32 range; the results of such a call are invalid and the caller repeats the step with
 * kgeb_fused_fwd + kgeb_fused_bwd (online maximum), as fused.AllEntityLoss and the steppers do.
 *   rowstat[B,4] = (mref, sum_e exp(x - mref), 0, sum of x over the row's labels in this shard)  -- kgeb_fused_fwd's layout,
 *                  i.e. kgeb_loss_from_rowstat and the shard combination (max + rescaled sums) apply unchanged
 *   o_sum[B,d]
 * Replaces K4 + K8 of SURVEY.md 2.3 (mm + log_softmax, distmult.py:20-22, loss.py:199-213) and the dQ half of their backward. */
int kgeb_fused_flash_fwd(const float* Q, int64_t B, int d, const float* table, int64_t e_lo, int64_t e_hi,
                         int64_t num_entities, const int64_t* lab_off, const int64_t* lab_col, int64_t nnz,
                         const void* table_bf16, float* rowstat, float* o_sum, int32_t* status, void* workspace,
                         int64_t workspace_bytes, void* stream);
/* dQ[q,:] = w_q * exp(mref_q - lse_q) * o_sum[q,:] - (w_q / nnz_q) * sum over the row's labels in this shard of table[e,:],
 * w_q = inv_batch * grad_scale[q] * (row q has labels).  rowstat_local = THIS shard's kgeb_fused_flash_fwd output (its
 * mref), lse = the global log-sum-exp (kgeb_loss_from_rowstat on the combined statistics).  No pass over the table. */
int kgeb_fused_flash_dq(const float* Q, int64_t B, int d, const float* table, int64_t e_lo, int64_t e_hi,
                        const int64_t* lab_off, const int64_t* lab_col, int64_t nnz, const float* rowstat_local,
                        const float* lse, float inv_batch, const float* grad_scale /* [B] or NULL */, const float* o_sum,
                        float* dQ, void* workspace, int64_t workspace_bytes, void* stream);
/* buf[0..numel) = 0 if *flag != 0 (any non-zero 32-bit word), else nothing.  Guard between the gradient computation and
 * the optimizer kernels of a captured step whose kgeb_fused_flash_fwd reported a failure: zero gradients make the Adagrad
 * kernels exact no-ops, the host then repeats the step with the two-pass kernels. */
int kgeb_zero_if(const int32_t* flag, float* buf, int64_t numel, void* stream);
/* What TrainingJobKvsAll logs per batch (train.py:744-747: avg_loss is overwritten once per query type, so the value of
 * the LAST non-empty query type survives): rows_loss[B] from kgeb_loss_from_rowstat, row_type[B] (0 = sp_, 1 = _po);
 * out[0] = sum of all rows (the cost that was back-propagated), out[1] = sum over the rows of the highest type present. */
int kgeb_loss_report(const float* rows_loss, const int32_t* row_type, int64_t B, float* out, void* stream);
/* Same for a reciprocal relations model whose _po rows were rewritten to sp_ rows on relation p + R (the *_inv batch
 * builders): a row counts as _po when row_type != 0 or p_idx[row] >= inv_rel_offset (> 0).  inv_rel_offset = 0 (p_idx
 * may be NULL) is kgeb_loss_report. */
int kgeb_loss_report_inv(const float* rows_loss, const int32_t* row_type, const int64_t* p_idx, int64_t inv_rel_offset,
                         int64_t B, float* out, void* stream);
/* fp32 -> bf16 (round to nearest even) mirror of a table / query matrix for KGEB_MATH_BF16 */
int kgeb_to_bf16(const float* src, void* dst, int64_t numel, void* stream);
int64_t kgeb_fused_workspace_bytes(int64_t B, int d, int64_t num_shard_entities, int64_t nnz);

/* ---- a23-a26/K10: fused score-and-count for filtered entity ranking (entity_ranking.py:153-217,
 * 469-529).  Q is [nq,d] (callers stack the B sp_ queries and the B _po queries).  For query i the
 * candidate true_ent[i] takes the precomputed true_score[i] (entity_ranking.py:170-177); NaN -> -inf
 * on both sides; filt CSR (offsets int64 [nq+1], cols int64 ascending per row) lists known answers of
 * the filter splits, test CSR those of the test split (may be NULL); the row's own true entity is
 * never filtered (entity_ranking.py:189-193); filters are cumulative (208-210).
 * counts[i*6 + {0,1}] = (rank, ties) raw, {2,3} filtered, {4,5} filtered-with-test; int64, ADDED to
 * the existing contents so that entity shards / chunks accumulate. */
int kgeb_rank_count(int kind, int math, const float* Q, int64_t nq, int d, const float* table, int64_t e_lo,
                    int64_t e_hi, const float* true_score, const void* true_ent, int idx64,
                    const int64_t* filt_off, const int64_t* filt_col, const int64_t* test_off,
                    const int64_t* test_col, int64_t* counts, void* stream);

/* ---- a3/K3: deterministic sort-based segment scatter-add (autograd of nn.Embedding,
 * lookup_embedder.py:39-41,91-92).  rows[n,d] are summed per distinct idx in a fixed order (stable sort
 * by id, then chunked ordered partial sums) and ADDED into dense[vocab,d].
 * workspace from kgeb_scatter_workspace_bytes(n, d). */
int64_t kgeb_scatter_workspace_bytes(int64_t n, int d);
int kgeb_scatter_add_rows(const void* idx, int idx64, const float* rows, int64_t n, int d, float* dense,
                          int64_t vocab, void* workspace, int64_t workspace_bytes, void* stream);
/* same, with the sort hoisted out: perm[n] (int32) = stable argsort of idx, e.g. computed once by the collate that
 * built idx (the ids of a batch are known before the step).  The sums and their order are identical to
 * kgeb_scatter_add_rows, so the results are bit-identical. */
int kgeb_scatter_add_rows_perm(const void* idx, int idx64, const int32_t* perm, const float* rows, int64_t n, int d,
                               float* dense, int64_t vocab, void* workspace, int64_t workspace_bytes, void* stream);
/* sparse form (lookup_embedder.yaml sparse: True): returns distinct ids (ascending) + summed rows */
int kgeb_segment_reduce_rows(const void* idx, int idx64, const float* rows, int64_t n, int d,
                             int64_t* uniq_ids /*[n]*/, float* uniq_rows /*[n,d]*/, int64_t* num_uniq /*dev*/,
                             void* workspace, int64_t workspace_bytes, void* stream);

/* ---- a21/K11: optimizer steps with torch.optim semantics (util/optimizer.py:10-17).
 * Adagrad: g += wd*w; state += g*g; w -= clr * g / (sqrt(state) + eps), clr = lr/(1+(step-1)*lr_decay) */
int kgeb_adagrad_dense(float* W, float* state, const float* grad, const float* grad2 /* added to grad, or NULL */,
                       int64_t numel, float clr, float eps, float weight_decay,
                       void* bf16_mirror /* updated alongside W, or NULL */, void* stream);
/* the same with clr read from the device word *clr (see kgeb_fused_bwd_update_sched) */
int kgeb_adagrad_dense_sched(float* W, float* state, const float* grad, const float* grad2, int64_t numel, const float* clr,
                             float eps, float weight_decay, void* bf16_mirror, void* stream);
/* touched-rows-only Adagrad (equals the dense step when untouched rows have zero gradient and wd=0) */
int kgeb_adagrad_rows(float* W, float* state, const int64_t* row_ids, const float* row_grads,
                      const int64_t* num_rows_dev, int64_t max_rows, int d, float clr, float eps, void* stream);
/* Adam (torch.optim.Adam, amsgrad=False): bias corrections computed by the caller */
int kgeb_adam_dense(float* W, float* exp_avg, float* exp_avg_sq, const float* grad, int64_t numel, float lr,
                    float beta1, float beta2, float eps, float weight_decay, float bias_corr1, float bias_corr2,
                    void* stream);

/* ---- a28/8f-1: device-side CSR key lookup over KvsAllIndex arrays (indexing.py:36-55):
 * keys[K,2] sorted lexicographically (int64); for each query pair finds its row or -1. */
int kgeb_csr_lookup(const int64_t* keys, int64_t num_keys, const int64_t* query_pairs, int64_t n,
                    int64_t* row_out, void* stream);

/* ---- 8f-1: on-device batch construction from device-resident KvsAllIndex arrays.
 * kgeb_index_t = one index of the reference (indexing.py:8-98) on the device: keys [num_keys,2] sorted
 * lexicographically, offsets [num_keys+1], values; all int64. */
typedef struct {
  const int64_t* keys;
  int64_t num_keys;
  const int64_t* offsets;
  const int64_t* values;
} kgeb_index_t;

/* Filter CSR of an evaluation batch (EntityRankingJob._collate, entity_ranking.py:53-77; job/util.py:5-38): for the
 * triples (s,p,o)[B] and num_splits filter splits (host arrays of index descriptors, <= 4), source list
 * j = row * num_splits + k holds, for row < B, the known objects of (s,p) in split k and, for row >= B, the known
 * subjects of (p,o) of triple row-B.  count: src_row[j] = key row in that index or -1, len[j] = list length.
 * The caller turns len into positions pos[] (exclusive scan); fill copies the lists to col[pos[j]...] and/or writes
 * sort_keys = (row << 32) | value, whose ascending order is the per-row merged order the ranking kernel needs. */
int kgeb_filter_csr_count(const kgeb_index_t* sp_indexes, const kgeb_index_t* po_indexes, int num_splits, const void* s,
                          const void* p, const void* o, int idx64, int64_t B, int64_t* src_row /*[2B*num_splits]*/,
                          int64_t* len /*[2B*num_splits]*/, void* stream);
int kgeb_filter_csr_fill(const kgeb_index_t* sp_indexes, const kgeb_index_t* po_indexes, int num_splits, int64_t B,
                         const int64_t* src_row, const int64_t* pos, int64_t* col /* or NULL */,
                         int64_t* sort_keys /* or NULL */, void* stream);

/* KvsAll training batch (TrainingJobKvsAll collate, train.py:590-677) from example ids: id < sp.num_keys is the
 * sp-query of that key row of the sp index, the others are po-queries of row id - sp.num_keys.  count writes the
 * query rows in the layout of kgeb_query_build (a_idx = the entity of the key, p_idx = its relation, row_combine) and
 * the label counts; the caller scans them into lab_off[B+1]; fill writes the label entities to lab_col (capacity
 * entries; *overflow is set to 1 on the device when a batch does not fit). */
int kgeb_kvsall_batch_count(const kgeb_index_t* sp_index, const kgeb_index_t* po_index, const int64_t* example_ids,
                            int64_t B, int64_t* a_idx, int64_t* p_idx, int32_t* row_combine, int64_t* len, void* stream);
int kgeb_kvsall_batch_fill(const kgeb_index_t* sp_index, const kgeb_index_t* po_index, const int64_t* example_ids,
                           int64_t B, const int64_t* lab_off, int64_t capacity, int64_t* lab_col, int32_t* overflow,
                           void* stream);

/* The whole KvsAll batch in one call, straight into the static input buffers of the graph-captured step: count,
 * scan, fill (lab_col zero-padded to `capacity`) and the three stable argsorts a_perm[B], p_perm[B], lab_perm[capacity]
 * (int32) that kgeb_fused_bwd / kgeb_scatter_add_rows_perm take.  No host synchronisation, no allocation. */
int64_t kgeb_kvsall_build_workspace_bytes(int64_t B, int64_t capacity);
int kgeb_kvsall_batch_build(const kgeb_index_t* sp_index, const kgeb_index_t* po_index, const int64_t* example_ids,
                            int64_t B, int64_t capacity, int64_t num_entities, int64_t num_relations, int64_t* a_idx,
                            int64_t* p_idx, int32_t* row_combine, int64_t* lab_off, int64_t* lab_col, int32_t* a_perm,
                            int32_t* p_perm, int32_t* lab_perm, int32_t* overflow, void* workspace,
                            int64_t workspace_bytes, void* stream);
/* Reciprocal relations model (relation table of 2 R rows, reciprocal_relations_model.py:70-83): with inv_rel_offset = R > 0
 * every po-query (p, o) is written as the sp-query (o, p + R) -- a_idx = o, p_idx = p + R, row_combine = KGEB_SP_ -- with
 * the same labels, and p_perm is the stable argsort of the shifted ids.  inv_rel_offset = 0 is kgeb_kvsall_batch_build. */
int kgeb_kvsall_batch_build_inv(const kgeb_index_t* sp_index, const kgeb_index_t* po_index, const int64_t* example_ids,
                                int64_t B, int64_t capacity, int64_t num_entities, int64_t num_relations, int64_t* a_idx,
                                int64_t* p_idx, int32_t* row_combine, int64_t* lab_off, int64_t* lab_col, int32_t* a_perm,
                                int32_t* p_perm, int32_t* lab_perm, int32_t* overflow, void* workspace,
                                int64_t workspace_bytes, int64_t inv_rel_offset, void* stream);

/* The 1vsAll batch (train.py:1032-1062: an sp_ pass with label o and a _po pass with label s over the same triples) from
 * the [B, 3] int64 triples: the same eight arrays as kgeb_kvsall_batch_build, 2 B rows (sp_ rows first), one label per
 * row, 2 B <= 8192.  One block; meant as the first node of the captured step's graph, so that a training step of the
 * reference's TrainingJob1vsAll costs the host one H2D copy of the triples and one graph launch. */
int kgeb_onevsall_batch_build(const int64_t* triples, int64_t B, int64_t num_entities, int64_t num_relations, int64_t* a_idx,
                              int64_t* p_idx, int32_t* row_combine, int64_t* lab_off, int64_t* lab_col, int32_t* a_perm,
                              int32_t* p_perm, int32_t* lab_perm, void* stream);
/* Same with inv_rel_offset = R > 0: rows B..2B-1 are the sp_ queries (o, p + R) of a reciprocal relations model (label s,
 * row_combine = KGEB_SP_), p_perm sorts the shifted ids.  inv_rel_offset = 0 is kgeb_onevsall_batch_build. */
int kgeb_onevsall_batch_build_inv(const int64_t* triples, int64_t B, int64_t num_entities, int64_t num_relations,
                                  int64_t* a_idx, int64_t* p_idx, int32_t* row_combine, int64_t* lab_off, int64_t* lab_col,
                                  int32_t* a_perm, int32_t* p_perm, int32_t* lab_perm, int64_t inv_rel_offset, void* stream);

/* ---- 8f-2: on-device negative sampling (kge/util/sampler.py).  Philox4x32-10, counter-based: results depend only on
 * state = {seed, offset} (device memory, so CUDA-graph replays draw fresh numbers; kgeb_philox_advance bumps the offset
 * on the stream), never on launch shape.  The reference's torch / numpy / `random` streams cannot be reproduced on a
 * device; oracle/sampler_oracle.py restates THIS generator in numpy and the tests compare bit for bit. */
int kgeb_philox_words(uint64_t seed, uint64_t offset, uint64_t elem0, int64_t n, uint32_t* out /*[4n]*/, void* stream);
int kgeb_philox_advance(uint64_t* state, uint64_t inc, void* stream);
/* KgeUniformSampler._sample (sampler.py:195-198): out[i] uniform in [0, vocab), i < n = batch * num_samples */
int kgeb_sample_uniform(const uint64_t* state, int64_t vocab, int64_t n, int64_t* out, void* stream);
/* _filter_and_resample (sampler.py:148-176 / 257-315): row i's samples that occur among the known positives of its key
 * pair (key_a[i], key_b[i]) in `index` (the "<split>_<pair>_to_<slot>" index) are redrawn until they are true negatives.
 * *status is set to 1 when a row cannot be satisfied within 65536 redraws (the reference would loop forever). */
int kgeb_sample_filter(const uint64_t* state, int64_t vocab, const kgeb_index_t* index, const int64_t* key_a,
                       const int64_t* key_b, int64_t B, int64_t N, int64_t* negatives /*[B,N] in/out*/, int32_t* status,
                       void* stream);
/* KgeUniformSampler._sample_shared (sampler.py:200-255): one set of num_distinct+1 distinct samples shared by the batch;
 * each row drops its own positive if sampled, else a random position; WR upsamples to N columns.
 * meta[0] = num_distinct, meta[1] = 1 if the draw did not converge. */
int64_t kgeb_sample_shared_workspace_bytes(int64_t N);
int kgeb_sample_shared(const uint64_t* state, int64_t vocab, const int64_t* positives /*[B] slot column*/, int64_t B,
                       int64_t N, int with_replacement, int64_t* out /*[B,N]*/, int32_t* meta /*[2]*/, void* workspace,
                       int64_t workspace_bytes, void* stream);

/* ---- a22 / 8f-3: Lp penalties of LookupEmbedder (lookup_embedder.py:112-158) with their gradient, deterministic.
 * dense (unweighted):  value_out[0] = weight/p * sum |W|^p ;  grad += weight * |W|^(p-1) sign(W)  (grad may be NULL)
 * rows (weighted):     over the distinct indexes u (multiplicity c_u) of indexes[n]:
 *                      value_out[0] = weight/p * sum_u c_u sum_k |W[u,k]|^p / n ;  grad[u,:] += weight c_u/n |W|^(p-1) sign(W)
 * adagrad_dense_lp:    kgeb_adagrad_dense with the dense penalty gradient formed from the parameter it reads anyway
 *                      and value_out[0] = the penalty of the pre-update parameters (train.py:320-338 then :375). */
int64_t kgeb_penalty_workspace_bytes(int64_t n_indexes, int64_t numel);
int kgeb_lp_penalty_dense(const float* W, int64_t numel, int p, float weight, float* grad, float* value_out,
                          void* workspace, int64_t workspace_bytes, void* stream);
int kgeb_lp_penalty_rows(const float* W, int64_t vocab, int dim, const void* indexes, int idx64, int64_t n, int p,
                         float weight, float* grad, float* value_out, void* workspace, int64_t workspace_bytes,
                         void* stream);
int kgeb_adagrad_dense_lp(float* W, float* state, const float* grad, const float* grad2, int64_t numel, float clr,
                          float eps, float weight_decay, int p, float pen_weight, void* bf16_mirror, float* value_out,
                          void* workspace, int64_t workspace_bytes, void* stream);
/* the same with clr read from the device word *clr (see kgeb_fused_bwd_update_sched) */
int kgeb_adagrad_dense_lp_sched(float* W, float* state, const float* grad, const float* grad2, int64_t numel,
                                const float* clr, float eps, float weight_decay, int p, float pen_weight, void* bf16_mirror,
                                float* value_out, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- 8f-4: rank histograms and metrics on the device (eval.py:138-224, entity_ranking.py:553-577).
 * rank_hist:    hist[ranks[i]] += 1 for every i with mask[i] != 0 (mask NULL = all); *status = 1 on a rank outside
 *               [0, num_entities).  isin_sorted builds the drill-down masks (`id in set`, eval.py:187,205-221).
 * rank_metrics: out = {count, mean_rank, mean_reciprocal_rank, hits@k[0..num_k)} (double, device); hits_at_k is a
 *               HOST array of at most 16 values; all metrics 0 for an empty histogram. */
int kgeb_rank_hist(const int64_t* ranks, const uint8_t* mask, int64_t n, int64_t num_entities, float* hist,
                   int32_t* status, void* stream);
int kgeb_isin_sorted(const void* values, int idx64, int64_t n, const int64_t* sorted_set, int64_t m, uint8_t* mask,
                     void* stream);
int64_t kgeb_rank_metrics_workspace_bytes(void);
int kgeb_rank_metrics(const float* hist, int64_t num_entities, const int32_t* hits_at_k, int num_k, double* out,
                      void* workspace, int64_t workspace_bytes, void* stream);

/* One-shot all-reduce of a small fp32 buffer over peer-mapped (symmetric) memory, as a plain kernel that sits in the same
 * CUDA graph as the compute around it: the three O(batch * d) exchanges of the row-sharded all-entity step (SURVEY.md 8e:
 * query-side rows, row statistics, dQ).  peer_bufs[k] = rank k's partial (this rank's own partial is peer_bufs[rank]);
 * out (local) = reduction over the ranks in rank order (bit-identical everywhere).  mode 0: sum; mode 1: every 4 floats
 * are a row statistic (max, sum-exp relative to max, sum x, label dot) combined as log-sum-exp partials.  epoch = two
 * device words [barrier epoch, block ticket], zero-initialised, shared by all collectives of a stepper.  A buffer may be
 * rewritten after the NEXT collective on the same epoch counter has completed. */
int kgeb_p2p_allreduce(const void* const* peer_pads, const void* const* peer_bufs, int rank, int world, uint32_t* epoch,
                       uint32_t* timeout_flag, int64_t numel, int mode, float* out, void* stream);
/* ---- 8e (replicas row): data-parallel gradient exchange fused with the Adagrad update over NVLink peer memory.
 * All pointer arrays are HOST arrays of `world` device pointers, entry k = rank k's buffer mapped into this process
 * (torch symmetric memory / cuMem VMM + IPC).  Replaces  all-reduce(grad) ; torch.optim.Adagrad.step  (train.py:375)
 * of replicated training with two kernels per step, capturable in the step's CUDA graph:
 * p2p_exchange: [barrier: every rank's gradients are complete]  rank r reduces its slice of each table's gradient over
 *   all ranks in rank order, updates its slice of W / state / bf16 mirror and stores the new values into every peer's
 *   staging buffer; loss_out[0] = sum of the ranks' losses.  peer_flat[k] = rank k's [g_table0 | g_table1 | loss],
 *   peer_stage[k] = rank k's [W_table0 | W_table1] staging buffer.
 * p2p_apply:    [barrier: all pushes have landed]  copies the other owners' slices from the local staging buffer into
 *   the tables (+ mirror) and advances *ctr.
 * Signal pad of rank k = uint32[world] (zero-initialised); *ctr = completed steps (device, zero-initialised), the two
 * barriers of step s use the values 2s+1 and 2s+2; *ticket = 0; *timeout_flag is set if a peer does not arrive within
 * ~10 s (a dead peer must not hang the GPU). */
int kgeb_p2p_exchange(const void* const* peer_pads, const void* const* peer_flat, const void* const* peer_stage, int rank,
                      int world, const uint32_t* ctr, uint32_t* timeout_flag, float* W0, float* state0, void* mirror0,
                      int64_t numel0, float* W1, float* state1, int64_t numel1, float* loss_out, float clr, float eps,
                      void* stream);
/* the same with the rates read from device memory: clr[0] for table 0, clr[1] for table 1 (see
 * kgeb_fused_bwd_update_sched); every rank must hold the same words */
int kgeb_p2p_exchange_sched(const void* const* peer_pads, const void* const* peer_flat, const void* const* peer_stage,
                            int rank, int world, const uint32_t* ctr, uint32_t* timeout_flag, float* W0, float* state0,
                            void* mirror0, int64_t numel0, float* W1, float* state1, int64_t numel1, float* loss_out,
                            const float* clr, float eps, void* stream);
int kgeb_p2p_apply(const void* const* peer_pads, const float* stage, int rank, int world, uint32_t* ctr, uint32_t* ticket,
                   uint32_t* timeout_flag, float* W0, void* mirror0, int64_t numel0, float* W1, int64_t numel1,
                   void* stream);

/* One slot of a negative-sampling batch in one kernel (train.py:860-999, implementation "triple"; replaces
 * kgeb_pairs_score + kgeb_ns_loss + kgeb_pairs_bwd): cand int64 [B, M], column 0 = the positive.  Outputs dQ [B,d], row_loss
 * [B] (scaled by inv_batch) and the candidate gradient: dense == NULL -> rows dC [B*M, d] for the deterministic sorted
 * scatter; dense != NULL -> added to dense[cand, :] with vector reductions (no rows, no sort; order-dependent rounding:
 * the opt-in, not bit-reproducible fast path).  d % 4 == 0. */
int kgeb_ns_fused(int kind, int loss, const float* Q, const float* table, const int64_t* cand, int64_t B, int64_t M, int d,
                  float offset, float inv_batch, float* dQ, float* dC, float* dense, float* row_loss, void* stream);
/* ---- a20 (tuning path): negative-sampling backward without materialised candidate-gradient
 * rows.  ns_bwd_q = the dQ half of kgeb_pairs_bwd (no dC).  ns_cand_grad = the candidate half: pairs sorted by candidate
 * id (stable), one warp per distinct candidate recomputes its occurrences' rows from Q and adds their sum to
 * dense[vocab, d] -- replaces kgeb_pairs_bwd's dC output + kgeb_scatter_add_rows(cand, dC).  cand: int64 [B, M]. */
int kgeb_ns_bwd_q(int kind, const float* Q, const float* table, const int64_t* cand, int64_t B, int64_t M, int d,
                  const float* G, const float* scores, float* dQ, void* stream);
int64_t kgeb_ns_segment_workspace_bytes(int64_t n);
int kgeb_ns_cand_grad(int kind, const float* Q, const float* table, const int64_t* cand, int64_t B, int64_t M, int d,
                      const float* G, const float* scores, int64_t vocab, float* dense, void* workspace,
                      int64_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* KGEB200_H */
