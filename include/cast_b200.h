/* cast_b200.h — C ABI of the B200-native SASRec / CAST training-and-evaluation hot path.
 *
 * The reference (Spijkervet/Context-Aware-Sequential-Recommendation) has no FFI layer: its arithmetic lives in
 * TensorFlow-1.15 ops called from modules.py / models/*.py.  Each entry point below replaces the TF op group
 * cited next to it (paths relative to the reference root).  The Python model classes of this repo
 * (`SASRec`, `CAST1..9`, same constructor / predict protocol as models/sasrec.py:5,127) are the only callers.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer (fp32 / int32, row-major, contiguous unless an ld/stride is given);
 *   - `stream` is a cudaStream_t passed as void*; calls only enqueue work, never synchronise, allocate or free;
 *   - return value: CAST_OK (0) or a negative CAST_ERR_*; `cast_last_error_string()` explains the last failure;
 *   - scratch memory is caller-provided: `cast_<op>_workspace_bytes(...)` gives the size;
 *   - N = B*T rows ("positions"); H = hidden_units; h = num_heads; V = rows of an embedding table;
 *   - dropout is counter based: keep(site, idx) = hash(seed, *step, site, idx) >= rate*2^32, where idx is the
 *     flat element index in the reference's tensor layout, so backward kernels and tests regenerate identical
 *     masks (`cast_dropout_keep` materialises one).  `step` is a device pointer (may be null => 0) so a captured
 *     CUDA graph stays valid across steps.
 *   - all reductions run in a fixed order: results are bit-reproducible run to run.
 */
#ifndef CAST_B200_H_
#define CAST_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CAST_OK 0
#define CAST_ERR_BAD_ARG (-1)
#define CAST_ERR_UNSUPPORTED (-2)
#define CAST_ERR_WORKSPACE (-3)
#define CAST_ERR_CUDA (-4)

#define CAST_ABI_VERSION 1

int cast_version(void);
const char* cast_last_error_string(void);
/* number of kernels this library has enqueued so far in this process (each launch site counts once). */
unsigned long long cast_launch_count(void);
/* crc32c (Castagnoli) of a HOST buffer, continuing from crc_in (0 to start): the tensor checksum of the reference's
 * checkpoint format (tf.train.Saver tensor bundles, main.py:153-159,226-228). */
unsigned int cast_crc32c(const void* data, size_t n, unsigned int crc_in);

/* modules.py:148-160 `embedding` (zero-padded row 0, x sqrt(H)) + position row add (sasrec.py:39-56) + context
 * add (cast_1.py:87) + tf.layers.dropout (sasrec.py:59) + `*= mask` (sasrec.py:62).
 * out[n,:] = ((ids[n] ? table[ids[n],:]*scale : 0) + pos[n % T,:] + add[n,:]) * dropout * (mask_ids[n] != 0)
 * pos / add / mask_ids may be null; drop_rate 0 disables dropout. */
int cast_embed_fwd(const int* ids, const float* table, int V, int H, long N, int T, float scale, const float* pos,
                   const float* add, float drop_rate, unsigned long long seed, const unsigned long long* step,
                   int site, const int* mask_ids, float* out, void* stream);

/* ---- row-sharded item table (BASELINE config 5, SURVEY §8e): ownership is cyclic, item id -> rank id % n, local row
 * id / n (+1 on ranks 1..n-1, whose local row 0 is a pad, so that "row 0 is not an item" holds on every shard).
 * `shards` is a DEVICE array of n device pointers to the ranks' [rows_per_shard, H] shards (own shard + peer mappings
 * read over NVLink, cast_peer_open).  The *_sharded gathers are otherwise identical to their namesakes. */
int cast_embed_fwd_sharded(const int* ids, const float* const* shards, int nshards, int V, int H, long N, int T,
                           float scale, const float* pos, const float* add, float drop_rate, unsigned long long seed,
                           const unsigned long long* step, int site, const int* mask_ids, float* out, void* stream);
int cast_logits_loss_sharded(const float* seq_emb, const float* const* shards, int nshards, int V, int H, long N,
                             const int* pos, const int* neg, float* pos_logits, float* neg_logits, float* sums,
                             float* dseq, float* gpos, float* gneg, void* workspace, size_t workspace_bytes,
                             void* stream);
int cast_score_rank_cand_sharded(const float* seq_last, long ld, const float* const* shards, int nshards, int V, int H,
                                 long U, const int* cand, int C, float* logits, int* count_greater, int* count_equal,
                                 void* stream);
/* Embedding-gradient exchange without a table collective: every rank sorts its (id, entry) pairs by owner-major key
 * (cast_scatter_sort_sharded) and leaves the sorted arrays + its source rows in memory its peers can read; every owner
 * then folds, rank by rank in rank order, the entries that belong to its rows into its dense gradient shard
 * (cast_scatter_apply_range; keys of rank r: [r*rows_per_shard, (r+1)*rows_per_shard)).  cast_scatter_sorted_offsets
 * locates the sorted arrays inside a sort workspace. */
/* tuning hook: sorted entries walked by one warp in the segment sums (32 or 64; 0 = per call from the mean run length) */
int cast_scatter_set_chunk(int entries);
int cast_scatter_sort_sharded(const int* keys, int nsrc, long N, int V, int nshards, int rows_per_shard,
                              void* workspace, size_t workspace_bytes, void* stream);
int cast_scatter_sorted_offsets(long N, int nsrc, int Vkeys, size_t* keys_offset, size_t* payload_offset);
int cast_scatter_apply_range(int nsrc, long N, const float* const* rows, const float* const* rowscale,
                             const float* scale, int H, float* dtable, const void* sorted_keys,
                             const void* sorted_payload, unsigned key_lo, unsigned key_hi, void* partial,
                             size_t partial_bytes, int accumulate, void* stream);
/* cast_scatter_apply_range for a PEER's entries: its in-range rows are first gathered (one warp per entry: thousands
 * of rows in flight over NVLink) into local staging of cast_scatter_stage_bytes, then summed locally; same arithmetic. */
size_t cast_scatter_stage_bytes(long N, int nsrc, int H);
int cast_scatter_pull_range(int nsrc, long N, const float* const* rows, const float* const* rowscale,
                            const float* scale, int H, float* dtable, const void* sorted_keys,
                            const void* sorted_payload, unsigned key_lo, unsigned key_hi, void* stage,
                            size_t stage_bytes, void* partial, size_t partial_bytes, int accumulate, void* stream);
/* Peer memory (CUDA IPC).  cast_peer_alloc: a zeroed device allocation other processes of the box may map, and its
 * 64-byte cudaIpcMemHandle; cast_peer_open maps a peer's allocation into this process with peer access enabled and
 * returns its base pointer (one open per handle and process); both are setup-time calls (they synchronise). */
int cast_peer_alloc(size_t bytes, void** ptr, void* ipc_handle64);
int cast_peer_free(void* ptr);
int cast_peer_open(const void* ipc_handle64, void** base_ptr);
int cast_peer_close(void* base_ptr);
/* Gradient exchange of data-parallel training over peer memory (no collective library in the step; everything below is
 * a plain kernel launch, so the whole step is one CUDA graph): cast_peer_barrier = flag barrier over NVLink (flags:
 * DEVICE array of n pointers to the ranks' n x u64 arrival arrays; state: this rank's {epoch, timed-out flag});
 * cast_peer_reduce: out[i] = sum over ranks, in rank order, of grads[r][i] — the same bits on every rank. */
int cast_peer_barrier(void* const* flags, int rank, int n, void* state, void* stream);
int cast_peer_reduce(const void* const* grads, int n, long count, float* out, void* stream);

/* element-wise backward of `x -> dropout(x) * mask`: out_masked = in*mask, out_masked_dropped = in*mask*dropout
 * (either output may be null).  Used for sasrec.py:59-62 and modules.py:307-311 backward. */
int cast_mask_dropout(const float* in, const int* mask_ids, float drop_rate, unsigned long long seed,
                      const unsigned long long* step, int site, long N, int H, float* out_masked,
                      float* out_masked_dropped, void* stream);

/* tf.concat(axis=2) + tf.layers.dropout of the CAST merges (cast_2.py:89-92, cast_4.py:114-124):
 * cat[n, s*H+c] = srcs[s][n,c] * dropA(first width_a sources, index in the [N, width_a*H] tensor)
 *                              * dropB(all k sources, index in the [N, k*H] tensor).  k <= 4. srcs is a HOST array. */
int cast_concat_dropout_fwd(const float* const* srcs, int k, int width_a, long N, int H, float rate_a, int site_a,
                            float rate_b, int site_b, unsigned long long seed, const unsigned long long* step,
                            float* cat, void* stream);
int cast_concat_dropout_bwd(const float* dcat, int k, int width_a, long N, int H, float rate_a, int site_a,
                            float rate_b, int site_b, unsigned long long seed, const unsigned long long* step,
                            float* const* dsts, void* stream);

/* keep[i] = 1 if element i of dropout site `site` is kept (test / oracle hand-off helper). */
int cast_dropout_keep(float drop_rate, unsigned long long seed, const unsigned long long* step, int site, long n,
                      unsigned char* keep, void* stream);

int cast_add(const float* a, const float* b, float* out, long n, void* stream);
/* out = dy * (act > 0 ? scale : 0): backward of tf.nn.relu in `mlp` (modules.py:333-334). */
int cast_relu_bwd(const float* dy, const float* act, float scale, float* out, long n, void* stream);

/* modules.py:53-80 `normalize`: y = gamma*(x-mean)/sqrt(var_biased+eps)+beta.  Optionally saves mean / rstd and the
 * flags xnz[n] = (sum_H x[n,:] != 0), ynz[n] = (sum_H y[n,:] != 0) that multihead_attention turns into its key
 * mask (modules.py:222) and query mask (modules.py:248). */
int cast_layernorm_fwd(const float* x, const float* gamma, const float* beta, long N, int H, float eps, float* y,
                       float* mean, float* rstd, float* xnz, float* ynz, void* stream);
size_t cast_layernorm_bwd_workspace_bytes(long N, int H);
/* dx = LN'(dy) (+ dx_add if non-null); dgamma, dbeta overwritten (deterministic two-stage reduction). */
int cast_layernorm_bwd(const float* dy, const float* x, const float* mean, const float* rstd, const float* gamma,
                       long N, int H, const float* dx_add, float* dx, float* dgamma, float* dbeta, void* workspace,
                       size_t workspace_bytes, void* stream);

/* tf.layers.dense / conv1d(k=1) (modules.py:203-205, :298-306, :333-334) and their gradients as one strided GEMM:
 *   C[i,j] = epi( sum_k A[i*sam + k*sak] * B[k*sbk + j*sbn] ),  i<M, j<N, k<K
 *   epi(c) = (((relu?max(c+bias[j],0):c+bias[j]) * dropout(i*N+j)) * (act[i,j]>0 ? act_scale : 0) + resid[i,j])
 *            * (row_ids[i] != 0)                      — every term optional (null / 0).
 * splits > 1: reduction dimension split across CTAs, partials summed in fixed order (no epilogue, ldc == N). */
/* Backends: shapes with M, N, K >= 64 and M*N*K >= 2.5e8 run on the tensor cores (tcgen05.mma kind::tf32, 3xTF32 operand split,
 * accumulator in TMEM — csrc/gemm_umma.cu), smaller ones on FP32 FFMA register tiles (csrc/gemm.cu).
 * cast_gemm_set_backend: 0 = that rule, 1 = always FFMA, 2 = always tensor cores (tests).
 * (The TMEM accumulator rounds toward zero; reductions longer than ~1k per CTA should use splits > 1.)
 * cast_gemm_tensor_status synchronises the stream and returns the tensor path's watchdog flag (0 = ok). */
int cast_gemm_set_backend(int which);
int cast_gemm_tensor_status(int* host_flag, void* stream);
size_t cast_gemm_workspace_bytes(long M, int N, long K, int splits);
int cast_gemm(const float* A, long sam, long sak, const float* B, long sbk, long sbn, float* C, long ldc, long M,
              int N, long K, const float* bias, int relu, float drop_rate, unsigned long long seed,
              const unsigned long long* step, int site, const float* act, long ld_act, float act_scale,
              const float* resid, long ldr, const int* row_ids, int splits, void* workspace, size_t workspace_bytes,
              void* stream);

/* ---- fused row-tile kernels of one transformer block, hidden_units <= 64 (cast_fused_supported) -------------------
 * ln_qkv_fwd  = normalize (modules.py:74-78) + the three tf.layers.dense of multihead_attention (:203-205) + the key /
 *               query zero-sum flags (:222, :248).
 * ln_ffn_fwd  = normalize + feedforward (modules.py:298-313) + `*= mask` (sasrec.py:83); saves LN output zn, the
 *               post-dropout hidden activation h1d, LN stats.
 * ffn_bwd / qkv_bwd = their backward passes.  Parameter gradients are written to `grads_out`, which must be the
 *               contiguous flat block  [ln.beta H | ln.gamma H | W H*H | b H | ...]  in the order
 *               (ffn_bwd) ln2.beta, ln2.gamma, ffn1.w, ffn1.b, ffn2.w, ffn2.b
 *               (qkv_bwd) ln1.beta, ln1.gamma, q.w, q.b, k.w, k.b, v.w, v.b          (all W stored [in,out]).
 *               qkv_bwd adds `dres` (gradient of the `outputs += queries` residual, modules.py:269) to d(LN(x)). */
int cast_fused_supported(int H);
int cast_ln_qkv_fwd(const float* x, const float* gamma, const float* beta, const float* Wq, const float* bq,
                    const float* Wk, const float* bk, const float* Wv, const float* bv, long N, int H, float eps,
                    float* qn, float* Q, float* K, float* V, float* mean, float* rstd, float* kmask, float* qmask,
                    void* stream);
int cast_ln_ffn_fwd(const float* y, const float* gamma, const float* beta, const float* W1, const float* b1,
                    const float* W2, const float* b2, const int* ids, float drop_rate, unsigned long long seed,
                    const unsigned long long* step, int site_hidden, int site_out, long N, int H, float eps, float* zn,
                    float* h1d, float* xout, float* mean, float* rstd, void* stream);
/* ---- the same forward row kernels on the 5th-generation tensor cores (tcgen05.mma kind::tf32, TMEM accumulators) -----
 * cast_rowk_supported(H): hidden_units the tcgen05 row kernels accept (their shared-memory plan must fit 227 KB).
 * cast_rowk_presplit: once per step (weights change with every Adam update), splits the five [H,H] matrices of each
 *   block {Wq, Wk, Wv, W1, W2} (`weights` = HOST array of nblocks*5 device pointers) into tf32 hi/lo operand images
 *   (K-major UMMA layout; transposed and plain forms) at images + b * cast_rowk_image_bytes(H).
 * cast_rowk_ln_qkv_fwd / cast_rowk_ln_ffn_fwd: same contract as cast_ln_qkv_fwd / cast_ln_ffn_fwd, weights taken from
 *   the block's images.  cast_rowk_status reports (and clears) the kernels' barrier watchdog; it synchronises. */
int cast_rowk_supported(int H);
size_t cast_rowk_image_bytes(int H);
int cast_rowk_presplit(const float* const* weights, int nblocks, int H, void* images, size_t image_bytes, void* stream);
int cast_rowk_ln_qkv_fwd(const float* x, const float* gamma, const float* beta, const float* bq, const float* bk,
                         const float* bv, const void* images, long N, int H, float eps, float* qn, float* Q, float* K,
                         float* V, float* mean, float* rstd, float* kmask, float* qmask, void* stream);
int cast_rowk_ln_ffn_fwd(const float* y, const float* gamma, const float* beta, const float* b1, const float* b2,
                         const void* images, const int* ids, float drop_rate, unsigned long long seed,
                         const unsigned long long* step, int site_hidden, int site_out, long N, int H, float eps,
                         float* zn, float* h1d, float* xout, float* mean, float* rstd, void* stream);
int cast_rowk_status(int* timed_out);
/* test / tuning hook: cap the persistent grid (default and maximum: one CTA per SM) */
int cast_rowk_set_grid(int max_ctas);
/* tuning hook: device buffer of 148*4*16 int64 filled with clock64() phase stamps by the row kernels (NULL: off) */
int cast_rowk_set_trace(void* device_buffer);
/* Row-kernel backend (A/B testing): bit 0 = backward kernels on the tensor cores (mma.sync 3xTF32), bit 1 = forward
 * kernels; default 3; 0 = FP32 FFMA kernels. */
int cast_fused_set_backend(int backend);
size_t cast_block_bwd_workspace_bytes(long N, int H);
/* cast_ffn_bwd / cast_qkv_bwd sum their per-CTA gradient partials (workspace layout [parts][count], count =
 * 2H + 2(H*H+H) resp. 2H + 3(H*H+H)) into grads_out with a fixed-order reduction launch.  With grads_out == NULL the
 * partials are left in the workspace: the caller folds the partials of all blocks of a step in one launch with
 * cast_reduce_partials_batch (same fixed order, same bits).  cast_block_bwd_parts = number of partial blocks
 * (which: 0 = ffn_bwd, 1 = qkv_bwd). */
int cast_block_bwd_parts(long N, int which);
 /* out_j[c] = sum_{p < nparts_j} partials_j[p * pitch_j + c], c < count_j (pitches == NULL: pitch = count). */
int cast_reduce_partials_batch(int njobs, const float* const* partials, const int* nparts, const long* counts,
                               const long* pitches, float* const* outs, void* stream);
/* cast_layernorm_bwd with dgamma == dbeta == NULL leaves its partials [parts][gamma H | beta H] in the workspace. */
int cast_layernorm_bwd_parts(long N);
int cast_ffn_bwd(const float* dx, const int* ids, const float* zn, const float* h1d, const float* y, const float* mean,
                 const float* rstd, const float* gamma, const float* W1, const float* W2, float drop_rate,
                 unsigned long long seed, const unsigned long long* step, int site_out, long N, int H, float* dy,
                 float* grads_out, void* workspace, size_t workspace_bytes, void* stream);
int cast_qkv_bwd(const float* dQ, const float* dK, const float* dV, const float* dres, const float* x, const float* qn,
                 const float* mean, const float* rstd, const float* gamma, const float* Wq, const float* Wk,
                 const float* Wv, long N, int H, float* dx, float* grads_out, void* workspace, size_t workspace_bytes,
                 void* stream);
/* Block 0 of a tower whose input is dropout(embedding) * mask (sasrec.py:58-62): the same kernel, with dx also
 * multiplied by the padding mask of mask_ids (may be NULL) and the dropout keep/scale of (drop_rate, seed, *step, site)
 * at flat index row*H + col — i.e. cast_qkv_bwd followed by cast_mask_dropout, one launch, same bits. */
int cast_qkv_bwd_embed(const float* dQ, const float* dK, const float* dV, const float* dres, const float* x,
                       const float* qn, const float* mean, const float* rstd, const float* gamma, const float* Wq,
                       const float* Wk, const float* Wv, long N, int H, const int* mask_ids, float drop_rate,
                       unsigned long long seed, const unsigned long long* step, int site, float* dx, float* grads_out,
                       void* workspace, size_t workspace_bytes, void* stream);

/* out[c] = sum_r X[r*ld + c] (bias gradients; learned-position gradient = sum over the batch), deterministic. */
size_t cast_colsum_workspace_bytes(long rows, long cols);
int cast_colsum(const float* X, long rows, long cols, long ld, float* out, void* workspace, size_t workspace_bytes,
                void* stream);

/* modules.py:208-269: scaled QK^T, key mask, causal mask, softmax, query mask, dropout, PV, head merge, + queries.
 * Q,K,V: [B*T, ld]; queries = LN(x) [B*T,H] (residual); kmask/qmask: [B*T] 0/1 floats from cast_layernorm_fwd.
 * out [B*T,H]; attn_weights (optional) [h*B,T,T] = reference `attention_weights` (post dropout, modules.py:259);
 * row_max/row_linv (optional, needed for backward) [B,h,T].
 * skip_ids (optional) [B*T] item ids: the leading rows of a sequence whose id is 0 are padding whose block output is
 * multiplied by 0 afterwards (`seq *= mask`, sasrec.py:83); with skip_ids given (and attn_weights null) their
 * attention rows are not computed (out = queries there) and the backward pass gives them zero gradient. */
int cast_attn_fwd(const float* Q, long ldq, const float* K, long ldk, const float* V, long ldv, const float* queries,
                  const float* kmask, const float* qmask, int B, int T, int H, int h, float drop_rate,
                  unsigned long long seed, const unsigned long long* step, int site, const int* skip_ids, float* out,
                  float* attn_weights, float* row_max, float* row_linv, void* stream);
/* Tuning hook: columns per streamed chunk of the tensor-core attention kernels (32 or 64; default 32). */
/* Programmatic dependent launch of the training step's main-chain kernels.  Off (0, the default): ordinary
 * stream-ordered launches, any operand may come from the immediately preceding launch.  On (1, what engine.py sets):
 * the next kernel's CTAs may be scheduled while the previous kernel drains, and a kernel reads a few operands BEFORE it
 * waits (griddepcontrol.wait) for that previous kernel — the caller promises that those operands were complete earlier:
 *   - weights, biases, LayerNorm gamma / beta and the pre-split weight images of every row kernel;
 *   - cast_qkv_bwd(_embed): dQ, x, qn (only dK, dV and dres may be outputs of the immediately preceding launch);
 *   - cast_ffn_bwd: zn, h1d, y (only dx may be);
 *   - cast_attn_bwd with out / queries: every input except dO (Q, K, V, out, queries, masks, row_max, row_linv, skip_ids).
 * Everything else is read, and everything is written, after the wait, so results do not change. */
int cast_set_pdl(int on);
int cast_attn_set_chunk(int columns);
/* Tuning hook: warps that share one 16-row block of a 64-row attention tile, each taking a 32-key slice of every
 * streamed chunk (forward and dQ kernels): 2 = 8 warps, two CTAs per SM (default); 4 = 16 warps, one CTA per SM. */
int cast_attn_set_kg(int key_groups);
/* Gradient of the attention output (without the residual branch) w.r.t. Q, K, V.  rowD: scratch [B,h,T].
 * out / queries (optional, both or neither): the forward call's `out` and `queries`; with them (and d = H/h <= 64)
 * the tensor-core kernels run and D_i = sum_j P_ij dP_ij is taken as dO_i . (out_i - queries_i).
 * workspace (optional, cast_attn_bwd_workspace_bytes = 2 * B*h*T*T floats): the dQ kernel stores P~ and dS there and
 * the dK/dV kernel reads them back instead of recomputing the scores. */
size_t cast_attn_bwd_workspace_bytes(int B, int T, int h);
int cast_attn_bwd(const float* Q, long ldq, const float* K, long ldk, const float* V, long ldv, const float* dO,
                  const float* kmask, const float* qmask, const float* row_max, const float* row_linv,
                  const int* skip_ids, float* rowD, int B, int T, int H, int h, float drop_rate,
                  unsigned long long seed, const unsigned long long* step, int site, float* dQ, long lddq, float* dK,
                  long lddk, float* dV, long lddv, const float* out, const float* queries, void* workspace,
                  size_t workspace_bytes, void* stream);

/* Host-side training-batch sampler, stream-identical to the reference's sample_function (sampler.py:16-81) for a given
 * --seed: numpy's legacy RandomState (MT19937 + masked-rejection randint) restated in C++, consumed in the same order
 * (user draws until one with > 1 training events; negatives newest position first, rejecting the user's items).
 * user_ptr [usernum+2] is a CSR over user ids 0..usernum (user 0 empty) into items / ratings / hours / days / ts (the
 * latter four optional); edges / n_edges as in cast_time_features (optional).  cast_sampler_next fills [B,T] int32
 * arrays left-padded with zeros (timeseq / ratings / hours / days may be NULL).  The object owns host memory only. */
void* cast_sampler_create(int usernum, int itemnum, const long* user_ptr, const int* items, const int* ratings,
                          const int* hours, const int* days, const long long* ts, int maxlen, unsigned seed,
                          const long long* edges, int n_edges);
int cast_sampler_next(void* sampler, int B, int* user, int* seq, int* pos, int* neg, int* timeseq, int* ratings,
                      int* hours, int* days);
/* same stream; instead of the host-computed features the RAW int64 timestamps [B,T] of each window (0 = padding), for
 * cast_time_features on the device */
int cast_sampler_next_raw(void* sampler, int B, int* user, int* seq, int* pos, int* neg, long long* ts);
void cast_sampler_destroy(void* sampler);

/* Time-context ids from raw timestamps on the device (reference util.py:24-43 hour / weekday, util.py:73-120
 * get_timedelta_bin, applied per position by sampler.py:61-72 and util.py:276-289).  ts [B,T] int64 seconds, ids [B,T]
 * (0 = padding => all three outputs 0), ref [B] reference time per row or NULL (= ts[b,T-1], the newest event of the
 * left-padded row), edges[k] = smallest delta (seconds) whose bin exceeds k, tabulated on the host with the reference's
 * scalar rule (data.time_bin_edges): bin = #{k : edges[k] <= ref - ts}.  Outputs int32 [B,T]. */
int cast_time_features(const long long* ts, const long long* ref, const int* ids, int B, int T, const long long* edges,
                       int n_edges, int* bins, int* hours, int* days, void* stream);

/* models/sasrec.py:87-115: pos/neg row gathers from the zero-padded table, row dots, literal BCE
 * (-log(sigmoid+1e-24)), istarget mask, AUC.  sums[0..2] = {sum loss terms, sum auc terms, sum istarget}
 * (un-normalised: the caller divides, or all-reduces first under data parallelism, sasrec.py:105-108).
 * If dseq != null also writes d(sum loss)/dseq_emb [N,H] and the per-position logit gradients gpos/gneg [N]. */
size_t cast_logits_loss_workspace_bytes(long N);
int cast_logits_loss(const float* seq_emb, const float* table, int V, int H, long N, const int* pos, const int* neg,
                     float* pos_logits, float* neg_logits, float* sums, float* dseq, float* gpos, float* gneg,
                     void* workspace, size_t workspace_bytes, void* stream);
/* sums == NULL leaves the per-CTA partials [parts][3] in the workspace (folded later by cast_reduce_partials_batch). */
int cast_logits_loss_parts(long N);
/* Training tail in one launch (H <= 64): seq_emb = LayerNorm(x) (modules.py:53-80, the main tower's final normalize),
 * the logits / loss / AUC terms of cast_logits_loss on it, and dx = d(sum loss)/dx through that LayerNorm.
 * Workspace: [parts][3] loss partials followed by [parts][gamma H | beta H] LayerNorm-parameter partials, both left
 * for cast_reduce_partials_batch. */
int cast_lnf_loss_parts(long N);
size_t cast_lnf_loss_workspace_bytes(long N, int H);
int cast_lnf_loss(const float* x, const float* gamma, const float* beta, float eps, const float* table, int V, int H,
                  long N, const int* pos, const int* neg, float* seq_emb, float* pos_logits, float* neg_logits,
                  float* gpos, float* gneg, float* dx, void* workspace, size_t workspace_bytes, void* stream);

/* Deterministic sparse embedding gradient (TF autodiff of the gathers: unsorted_segment_sum, SURVEY a9):
 * dtable[r,:] = sum over entries e (in ascending e) with keys[e] == r of rows_s[n,:] * rowscale_s[n] * scale_s,
 * where e = s*N + n enumerates `nsrc` sources of N positions each; row 0 (zero pad) gets 0.  Implemented as a
 * stable LSD radix sort of (key, e) followed by a fixed-order segmented reduction (64-entry chunks per warp, chunk-
 * crossing runs stitched in chunk order): no float atomics, work per warp independent of id skew.
 * rows/rowscale/scale are HOST arrays of nsrc device pointers / floats (rowscale[s] may be null). */
size_t cast_scatter_workspace_bytes(long N, int nsrc, int V);     /* integer scratch (sort buffers) */
size_t cast_scatter_partial_bytes(long N, int nsrc, int H);       /* float scratch (chunk-crossing partial sums) */
/* The two halves of cast_scatter_rows: the sort depends on the ids only (run it early, e.g. on a side stream while the
 * forward pass computes), the apply consumes the sorted arrays left in `workspace`. */
int cast_scatter_sort(const int* keys, int nsrc, long N, int V, void* workspace, size_t workspace_bytes, void* stream);
int cast_scatter_apply(int nsrc, long N, const float* const* rows, const float* const* rowscale, const float* scale,
                       int V, int H, float* dtable, void* workspace, size_t workspace_bytes, void* partial,
                       size_t partial_bytes, int accumulate, void* stream);
/* accumulate != 0: dtable is not cleared and every touched row is added to (the sum over other sources left there by an
 * earlier cast_scatter_apply).  Measured at C2: running the pos/neg part on a side stream during backward and only the
 * input-embedding part at the end was slower (0.698 vs 0.666 ms/step: the side kernels take SMs from the persistent
 * backward kernels), so the engine keeps one apply over all three sources. */
int cast_scatter_rows(const int* keys /* [nsrc*N] */, int nsrc, long N, const float* const* rows,
                      const float* const* rowscale, const float* scale, int V, int H, float* dtable,
                      void* workspace, size_t workspace_bytes, void* partial, size_t partial_bytes, void* stream);

/* tf.train.AdamOptimizer(lr, beta1=.9, beta2=.98, eps=1e-8) (sasrec.py:120-121), dense on every element:
 *   g = grad/(*gdenom) + l2*w (gdenom: device scalar, e.g. the global sum(istarget); null => 1; l2 only for
 *   elements in [l2_lo, l2_hi));
 *   lr_t = lr*sqrt(1-b2p)/(1-b1p); m = b1*m+(1-b1)*g; v = b2*v+(1-b2)*g*g; w -= lr_t*m/(sqrt(v)+eps)
 * state = device {float b1p, float b2p, uint64 step}; after the update b1p*=b1, b2p*=b2, step+=1 (TF order). */
int cast_adam_init_state(void* state /* 16 bytes */, float beta1, float beta2, void* stream);
int cast_adam_tf_step(float* w, const float* grad, float* m, float* v, long n, float lr, float beta1, float beta2,
                      float eps, const float* gdenom, float l2, long l2_lo, long l2_hi, void* state, void* stream);
/* The same update on one contiguous range; advance != 0 steps the state afterwards.  A rank that owns a row shard of
 * the item table updates {its shard, the replicated weights} with two calls and advances once. */
int cast_adam_tf_range(float* w, const float* grad, float* m, float* v, long n, float lr, float beta1, float beta2,
                       float eps, const float* gdenom, float l2, long l2_lo, long l2_hi, void* state, int advance,
                       void* stream);

/* Data-parallel form of the same update (sasrec.py:105-121 with the global sum(istarget) as denominator): grads is a
 * DEVICE array of n_ranks device pointers (own buffer + peer mappings, cast_peer_open), each n + tail floats = gradient
 * numerators then [loss_sum, auc_sum, count, ...] (tail >= 3).  The update uses sum_r grads[r][i] taken in rank order
 * (same bits on every rank) divided by sum_r count_r; the reduced n + tail floats are also left in g_red.  One launch
 * instead of cast_peer_reduce + cast_adam_tf_step; bracket it with cast_peer_barrier like cast_peer_reduce. */
int cast_adam_tf_step_peers(float* w, const void* const* grads, int n_ranks, float* g_red, float* m, float* v, long n,
                            long tail, float lr, float beta1, float beta2, float eps, float l2, long l2_lo, long l2_hi,
                            void* state, void* stream);

/* sasrec.py:93-97 + util.py:318-321: logits[u,c] = seq_last[u,:] . table0[cand[u,c],:] (sequential-k, unfused
 * multiply/add so the order is reproducible), and for candidate 0 the pair (count_greater, count_equal_excl_self)
 * from which the reference rank follows (SURVEY A-12). */
int cast_score_rank_cand(const float* seq_last, long ld, const float* table, int V, int H, long U, const int* cand,
                         int C, float* logits, int* count_greater, int* count_equal, void* stream);

/* Full-catalog evaluation scoring (BASELINE north_star (4); the reference's util.py:291-321 only ever scores 101
 * candidates, its test_logits GEMM sasrec.py:93-97 is the same contraction over the whole table):
 *   count_greater[u] = #{ j in [1,V), j != target[u], j not in rated(u) : s(u,j) >  s(u,target[u]) }
 *   count_equal[u]   = #{ same set                                      : s(u,j) == s(u,target[u]) }
 * with s the canonical logit of cast_score_rank_cand (sequential-k, unfused fp32).  rank = count_greater.
 * seq_last [U, ld] last-position vectors; table [V,H] (row 0 = pad, never a candidate); rated_ptr [U+1] / rated_idx:
 * CSR of each user's already-seen item ids (unique per user; null => nothing excluded).
 * mode 0: tcgen05 tensor-core GEMM (3xTF32 split, accumulator in TMEM) + exact re-scoring of the error band;
 * mode 1: exact brute force.  Both return identical integers.  stats (optional, device, 2 x u64): [0] = number of
 * band candidates re-scored exactly.
 * target_score (optional, [U]): item-sharded evaluation (SURVEY §8e): `table` is this rank's row shard, `target` the
 * LOCAL row to leave out (0 when the target lives elsewhere) and its canonical score is handed in; the per-shard counts
 * of all ranks add up (one integer all-reduce) to the whole-catalog counts. */
size_t cast_score_rank_full_workspace_bytes(long U, int V, int H);
int cast_score_rank_full(const float* seq_last, long ld, const float* table, int V, int H, long U, const int* target,
                         const float* target_score, const int* rated_ptr, const int* rated_idx, int mode,
                         int* count_greater, int* count_equal, unsigned long long* stats, void* workspace,
                         size_t workspace_bytes, void* stream);
/* Synchronises the stream and reports the tensor-core pass's watchdog flag (0 = ok). */
int cast_score_rank_full_status(const void* workspace, long U, int V, int* host_flag, void* stream);

/* Exact full-catalog top-K recommendation.  For each user u (row u of seq_last, stride ld >= H): the K rows
 * j in [1, V) of `table` not in the user's exclusion row, ordered by the canonical logit (the fp32 dot of
 * cast_score_rank_cand: k ascending, multiply and add rounded separately) descending, then by row ascending;
 * top_scores are those logits bit for bit.  Fewer than K eligible rows: the tail is (0, -inf).  1 <= K <= 256.
 * excl_ptr [U+1] / excl_idx (optional CSR): per user, row ids in ascending order; ids outside [1, V) and duplicates
 * are ignored.  mode 0 = tcgen05 tensor cores as an exact filter (two passes + canonical re-scoring of the admitted
 * candidates; a user whose candidates overflow the buffer takes the exact path), mode 1 = exact brute force.  Both
 * modes return the same bits.  stats (optional, [2]): [0] candidates re-scored, [1] users on the exact fallback. */
size_t cast_topk_full_workspace_bytes(long U, int V, int H, int K);
int cast_topk_full(const float* seq_last, long ld, const float* table, int V, int H, long U, int K,
                   const int* excl_ptr, const int* excl_idx, int mode, int* top_ids, float* top_scores,
                   unsigned long long* stats, void* workspace, size_t workspace_bytes, void* stream);
/* Synchronises the stream and reports the tensor-core passes' watchdog flag (0 = ok). */
int cast_topk_full_status(const void* workspace, long U, int V, int H, int K, int* host_flag, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CAST_B200_H_ */
