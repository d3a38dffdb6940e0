/* sc_b200.h — C ABI of the B200-native ORT / ACORT captioning hot path.
 *
 * The reference (jiahuei/sparse-image-captioning) is pure Python/PyTorch and has no FFI of its own; its
 * boundary for this path is the Python class surface (SURVEY.md section 8b).  Each entry point below replaces
 * the ATen op sequence of the cited reference lines (paths relative to the reference checkout) and is what
 * the drop-in Python classes in sparse-image-captioning_b200/ bind through ctypes (see INTEGRATION.md).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless stated; the caller owns all memory; the library never allocates.
 *  - all work is enqueued on `stream` (CUDA-graph capturable); no host synchronisation inside.
 *  - return 0 on success, <0 for argument errors (codes below), >0 = cudaError_t of the failed launch.
 *    sc_last_error() returns a thread-local description.  No exceptions, no aborts.
 *  - dtype codes: SC_F32 = 0, SC_BF16 = 1.  Matrices are row-major.
 */
#ifndef SC_B200_H
#define SC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* sc_stream_t; /* == cudaStream_t */

#define SC_F32 0
#define SC_BF16 1

#define SC_OK 0
#define SC_ERR_SHAPE (-1)
#define SC_ERR_ALIGN (-2)
#define SC_ERR_DTYPE (-3)
#define SC_ERR_WORKSPACE (-4)
#define SC_ERR_UNSUPPORTED (-5)
#define SC_ERR_DRIVER (-6)

/* mask modes of the supermask layers (pruning/masked_layer.py:84-110, pruning/sampler.py:43-66) */
#define SC_MASK_NONE 0      /* weight used as is                                             */
#define SC_MASK_ROUND 1     /* eval:  W * rint(sigmoid(S))   (bit-exact: S > 1.5*2^-24)      */
#define SC_MASK_BERNOULLI 2 /* train: W * Bernoulli(sigmoid(S)), Philox4x32-10(seed, stream_id, element) */
#define SC_MASK_RAW 3       /* snip / mag_* / lottery_* / mask_freeze: W * S                 */
#define SC_MASK_UNIFORM 4   /* train with caller-provided uniforms: W * (u < sigmoid(S))     */

const char* sc_last_error(void);
int sc_version(void);

/* K1 / K3a — MaskedLinear.forward / nn.Linear on densified weights
 * (pruning/masked_layer.py:134-135; models/transformer.py:315-325 FFN ReLU; :345-358 residual).
 *   y[M,N] = epilogue( x[M,K] * (w (.) mask)[N,K]^T )      epilogue: +bias[N], ReLU, +residual[M,N] (fp32)
 * x_dtype = SC_BF16: tcgen05/TMEM tensor-core kernel; w is either bf16 (pre-masked, TMA-fed) or fp32 master
 *           weights + fp32 mask (mask applied in the operand-load prologue).  K % 8 == 0.
 * x_dtype = SC_F32 : fp32-FMA verification kernel (1e-5 parity mode); w fp32.
 * tile_n: 0 = auto, or 64/128/256 (tensor path).  residual may alias y. */
int sc_linear(const void* x, int x_dtype, const void* w, int w_dtype, const float* mask, int mask_mode,
              const float* uniforms, unsigned long long seed, unsigned long long stream_id, const float* bias,
              const float* residual, void* y, int y_dtype, int M, int N, int K, int relu, int tile_n,
              sc_stream_t stream);

/* K1 + K9 — LayerNorm folded around the tensor-core GEMM for inference (models/transformer.py:329-358:
 * x + dropout(sublayer(norm(x)))).  x, w bf16.
 *   consumer (ln_stats != NULL): w = (W (.) m) (.) a_2, ln_c[n] = sum_k w[n,k], bias = W b_2 + bias; x = bf16 copy of the
 *     un-normalised residual stream;  y = rstd * (x w^T) - rstd * mean * ln_c + bias, row statistics (unbiased std,
 *     1/(std+eps)) merged from ln_stats fp32 [M][K/32][2] = per 32-column chunk (sum, M2 about the chunk mean).
 *   producer (stats_out and/or y_bf16_copy != NULL): after bias / ReLU / residual the result goes to y (fp32), its bf16
 *     copy to y_bf16_copy and the chunk statistics of the stored rows to stats_out [M][N/32][2]. */
int sc_linear_ln(const void* x, const void* w, const float* bias, const float* residual, void* y, int y_dtype, int M, int N,
                 int K, int relu, int tile_n, const float* ln_stats, const float* ln_c, float ln_eps, void* y_bf16_copy,
                 float* stats_out, sc_stream_t stream);

/* Programmatic dependent launch (griddepcontrol) between consecutive kernels of a stream: 1 = on everywhere (default),
 * 0 = off; otherwise a mask: bit 0 = GEMM + inference kernels, bit 1 = training row / attention kernels, bit 2 = the GEMM
 * triggers its dependents as soon as its loads are issued (else implicitly at exit). */
int sc_set_pdl(int enabled);

/* K3b — the same product from CSR weights (rows = output features, 16-bit column indices, values in x's dtype).
 * The reference only stores the sparse form (pruning/prune.py:200-221). */
int sc_csr_spmm(const void* x, int dtype, const int* row_ptr, const unsigned short* col_idx, const void* vals,
                const float* bias, const float* residual, void* y, int y_dtype, int M, int N, int K, int relu,
                sc_stream_t stream);

/* K3b' — the same product from SLICED-ELL weights (slab = 32 output features, entry i of feature 32 s + l at
 * slab_ptr[s] + 32 i + l; slab widths are multiples of 4, padding entries are (column 0, value 0)).
 * x bf16: entries uint32 = (column << 16) | bf16 bits; x fp32: entries {uint32 column, fp32 value}.  K <= 6400. */
int sc_sell_spmm(const void* x, int dtype, const int* slab_ptr, const void* entries, const float* bias,
                 const float* residual, void* y, int y_dtype, int M, int N, int K, int relu, sc_stream_t stream);
/* K3b'' - the same product on the TENSOR CORES by gather (bf16 x [M, ldx], fp32 accumulate): per K chunk of 512 columns and group of
 * 8 output features, grp_ptr [chunks][groups + 1] points at 16-entry MMA steps of words (col_in_chunk << 19) | (feature_in_group
 * << 16) | bf16 bits (zero-valued padding words allowed).  The x slab is staged transposed in shared memory; ldmatrix gathers the
 * columns of a step as the A operand, the B operand (one non-zero per k slot) is built in registers.  Roofline: shared-memory
 * bandwidth, nnz x M x 2 bytes. */
int sc_gspmm(const void* x, int ldx, const int* grp_ptr, const void* entries, const float* bias, const float* residual, void* y,
             int y_dtype, int M, int N, int K, int relu, sc_stream_t stream);

/* K9 — LayerNorm a*(x-mean)/(std_unbiased+eps)+b (models/transformer.py:329-341).  x fp32 [rows,D]. */
int sc_layernorm(const float* x, const float* a, const float* b, void* y, int y_dtype, int rows, int D, float eps,
                 sc_stream_t stream);

/* K9 — MaskedEmbedding + InputEmbedding + PositionalEncoding:
 * out[r] = (table (.) mask)[tokens[r]] * scale + pe[pos0 + r % T]
 * (pruning/masked_layer.py:160-169; models/transformer.py:383-401). tokens int32. */
int sc_embed_pe(const int* tokens, const float* table, const float* mask, int mask_mode, const float* uniforms,
                unsigned long long seed, unsigned long long stream_id, const float* pe, void* out, int out_dtype,
                int rows, int D, int V, int T, int pos0, float scale, sc_stream_t stream);

/* K9 (LayerNorm-folded decode path) — the same embedding for pre-masked tables, emitting the fp32 residual stream, its
 * bf16 copy and the per-32-column (sum, M2) row statistics that sc_linear_ln consumes.  D % 32 == 0. */
int sc_embed_pe_stats(const int* tokens, const float* table, const float* pe, float* x32, void* x_bf16, float* stats, int rows,
                      int D, int V, int T, int pos0, float scale, sc_stream_t stream);

/* prune_weights / densify: out = w (.) mask  (pruning/prune.py:165-174) */
int sc_apply_mask(const float* w, const float* mask, int mask_mode, const float* uniforms, unsigned long long seed,
                  unsigned long long stream_id, void* out, int out_dtype, size_t n, sc_stream_t stream);

/* sum rint(sigmoid(S)) accumulated into *count_out (calculate_sparsities, pruning/prune.py:124-144, 249-252) */
int sc_mask_count(const float* logits, size_t n, unsigned long long* count_out, sc_stream_t stream);

int sc_cast_f32_bf16(const float* x, void* y, size_t n, sc_stream_t stream);
/* fused ingest (data/collate.py:107-112,196-216 -> device): y (bf16, device) = cast(pinned_host fp32), read over PCIe by the
 * kernel itself (the pinned buffer must be mapped, as cudaHostAlloc / torch pin_memory buffers are); ctas <= 0: 64 CTAs */
int sc_ingest_f32_bf16(const float* pinned_host, void* y, size_t n, int ctas, sc_stream_t stream);

/* pack_wrapper zero-padding of padded regions (utils/model_utils.py:149-168): x[r,:] *= (mask[r] != 0) */
int sc_mask_rows(float* x, const float* row_mask, int rows, int D, sc_stream_t stream);

/* K4 — BoxRelationalEmbedding + WG + ReLU + log + softmax attention + PV, fused
 * (models/relation_transformer.py:148-191, 196-256, 258-293).
 * q/k/v: element (row=b*N+i, head, d) at ptr[row*ld + head*dk + d]; boxes fp32 [B,N,4];
 * wg_w fp32 [h, 64 (trig) | 4], wg_b fp32 [h]; att_mask fp32 [B,N] or NULL. */
int sc_box_attention_fwd(const void* q, const void* k, const void* v, int ldq, int ldk, int ldv, int dtype,
                         const float* boxes, const float* wg_w, const float* wg_b, const float* att_mask, void* out,
                         int ldo, int B, int N, int h, int dk, int trig, float wave_len, sc_stream_t stream);

/* K4 (inference split) — the geometry bias of EVERY encoder layer from one evaluation of the sin/cos embedding
 * (models/relation_transformer.py:179-183, 196-256: the reference rebuilds emb[B,N,N,64] in each layer although it only
 * depends on the boxes).  wg_w fp32 [layers*h, 64 (trig) | 4], wg_b fp32 [layers*h];
 * bias fp32 [layers, B, h, N, N] = log(max(relu(WG . emb + b), 1e-6)). */
int sc_box_bias_all(const float* boxes, const float* wg_w, const float* wg_b, float* bias, int B, int N, int layers,
                    int h, int trig, float wave_len, sc_stream_t stream);

/* Same bias on the tensor cores (the bf16 inference path's encoder): [16 pairs, layers*h] = emb[16, 64] . WG^T as mma.sync tiles
 * with both operands split into bf16 hi + lo parts (three products, fp32 accumulation: ~1e-5 absolute on WG . emb), sin / cos /
 * log through the SFU after range reduction.  Trigonometric embedding only, layers*h a multiple of 8 (<= 64).  The exact kernel
 * above stays the fp32 verification / training path. */
int sc_box_bias_all_tc(const float* boxes, const float* wg_w, const float* wg_b, float* bias, int B, int N, int layers,
                       int h, float wave_len, sc_stream_t stream);

/* K4 (inference split) — box_attention given the bias of one layer (models/relation_transformer.py:258-293):
 * out = softmax(bias + masked_fill(QK^T/sqrt(dk), mask==0, -1e9)) V.  bf16, d_k = 64, N <= 128; one warp per
 * (image, head) on mma.sync tiles.  bias fp32 [B, h, N, N]; att_mask fp32 [B,N] or NULL. */
int sc_bias_attention_fwd(const void* q, const void* k, const void* v, int ldq, int ldk, int ldv, int dtype,
                          const float* bias, const float* att_mask, void* out, int ldo, int B, int N, int h, int dk,
                          sc_stream_t stream);

/* K5 — decoder self-attention, one new token per row, append-to-cache + attention
 * (models/transformer.py:230-295 incremental branch).  cache_[kv]: [slots][R][D]; anc: int32 [R, anc_ld]
 * ancestor row of slot s is anc[r][s / slot_div].  Attends slots [0,n_prev) + the new token; the new k,v are
 * stored in slot write_slot (skip with -1: reference quirk Q1). */
int sc_decode_self_attn_step(const void* q, const void* k, const void* v, int ldq, int ldk, int ldv, int dtype,
                             void* cache_k, void* cache_v, const int* anc, int anc_ld, int slot_div, void* out, int ldo,
                             int R, int D, int h, int n_prev, int write_slot, sc_stream_t stream);

/* K6 — decoder cross-attention step over the per-image memory K/V [B*N, ldm] (models/transformer.py:255-256). */
int sc_decode_cross_attn_step(const void* q, int ldq, const void* mem_k, const void* mem_v, int ldm, int dtype,
                              const float* att_mask, void* out, int ldo, int B, int beam, int N, int D, int h,
                              sc_stream_t stream);

/* K7 — log-softmax + beam_step + finished-beam handling of batch_beam_search, group_size 1
 * (models/caption_model.py:56-111, 151-226; utils/model_utils.py:121-146).
 * penalty_kind: 0 "", 1 "wu_<alpha>", 2 "avg_<alpha>".  seq/lp/anc are ping-pong buffers [B*beam, L].
 * Two launches: one CTA per (image, beam) row reads its logits row once (log-softmax statistics + the row's top-`beam`
 * candidates by final score), then one small CTA per image merges the rows and does the bookkeeping.
 * workspace: sc_beam_step_workspace_bytes(B, beam) bytes of device scratch, 16-byte aligned.
 * suppress_tok (optional int32 [B*beam], -1 = none): per-row token whose log-prob is -inf at this step (remove_bad_endings,
 * caption_model.py:161-168); penalized_col (>= 0): column whose log-prob is lowered by 1000 (suppress_UNK, :169-170);
 * both act after the normalisation, like the decoding constraint. */
int sc_beam_step_workspace_bytes(int B, int beam);
/* Generator fused with the row pass of the beam step (OutputEmbedding, models/transformer.py:405-413, + beam_step,
 * models/caption_model.py:56-111): the [M, N] logits are never written.  sc_linear_topk (bf16 x [M,K], bf16 w [N,K], fp32
 * bias) leaves per row sc_linear_topk_parts(N) records of 12 floats {max, sum exp(x - max), 5 largest logits, their
 * columns as int bits; only the first `candidates` (<= 5, = the beam size) are filled} in partials [M][parts][12];
 * sc_beam_step_partials reduces them to the log-softmax statistics and the
 * row candidates and then runs the same per-image merge / bookkeeping as sc_beam_step (temperature 1, no decoding
 * constraint, beam <= 5). */
int sc_linear_topk_parts(int N);
int sc_linear_topk(const void* x, const void* w, const float* bias, int M, int N, int K, float* partials, int candidates,
                   sc_stream_t stream);
int sc_beam_step_partials(const float* partials, int parts_per_row, int B, int beam, int V, int L, int t, int eos, int pad,
                          int penalty_kind, float penalty_alpha, const int* seq_in, int* seq_out, const float* lp_in,
                          float* lp_out, float* sum, const int* anc_in, int* anc_out, int* tokens_out, int* done_seq,
                          float* done_lp, double* done_p, int* done_count, void* workspace, size_t workspace_bytes,
                          sc_stream_t stream);
int sc_beam_step(const float* logits, int B, int beam, int V, int L, int t, int eos, int pad, float temperature,
                 int decoding_constraint, int penalty_kind, float penalty_alpha, const int* suppress_tok, int penalized_col,
                 const int* seq_in, int* seq_out,
                 const float* lp_in, float* lp_out, float* sum, const int* anc_in, int* anc_out, int* tokens_out,
                 int* done_seq, float* done_lp, double* done_p, int* done_count, void* workspace, size_t workspace_bytes,
                 sc_stream_t stream);
/* Diverse beam search (group_size G > 1, caption_model.py:30-226 with add_diversity :33-52): the beam step of group `group`
 * (its bdash = `beam` beams per image) at its local step t.  Candidates are ranked by sum + (log-prob - diversity_lambda *
 * count), count = the number of beams of groups p < group whose token at position t of their CURRENT history is that column;
 * the running sum and the finished-beam score take the penalised value, the stored per-token log-prob (lp_out, done_lp) the
 * unpenalised one.  group_seq: every group's seq ping-pong buffers as one int32 [G][2][B*beam][L] tensor (seq_in / seq_out
 * are two of them); the groups are staggered in time, so group p has run its local step min(t + group - p, L-1) already and
 * its current history is buffer (that step + 1) % 2.  Everything else as sc_beam_step / sc_beam_step_partials; group * beam
 * <= 256, and for the records path (group + 1) * beam <= 5 with sc_linear_topk candidates >= (group + 1) * beam. */
int sc_beam_step_diverse(const float* logits, int B, int beam, int V, int L, int t, int eos, int pad, float temperature,
                         int decoding_constraint, int penalty_kind, float penalty_alpha, const int* suppress_tok, int penalized_col,
                         const int* group_seq, int group, float diversity_lambda, const int* seq_in, int* seq_out,
                         const float* lp_in, float* lp_out, float* sum, const int* anc_in, int* anc_out, int* tokens_out,
                         int* done_seq, float* done_lp, double* done_p, int* done_count, void* workspace, size_t workspace_bytes,
                         sc_stream_t stream);
int sc_beam_step_partials_diverse(const float* partials, int parts_per_row, int B, int beam, int V, int L, int t, int eos, int pad,
                                  int penalty_kind, float penalty_alpha, const int* group_seq, int group, float diversity_lambda,
                                  const int* seq_in, int* seq_out, const float* lp_in, float* lp_out, float* sum,
                                  const int* anc_in, int* anc_out, int* tokens_out, int* done_seq, float* done_lp, double* done_p,
                                  int* done_count, void* workspace, size_t workspace_bytes, sc_stream_t stream);

/* greedy branch of _generate_captions (models/transformer.py:507-561) */
int sc_greedy_step(const float* logits, int R, int V, int L, int t, int eos, int decoding_constraint, int* seq,
                   float* seq_lp, int* tokens, int* unfinished, int* live_count, sc_stream_t stream);
/* multinomial step (num_random_sample > 0, models/transformer.py:531-538): token ~ Categorical(exp(log_softmax(x) / T)) by
 * inverse CDF in index order with u = uniforms[r] (fp32 [R], tests) or Philox(seed, stream t, row r) when uniforms == NULL
 * (seed: immediate, or bit 63 set = device pointer to the 64-bit seed, so a captured graph can be re-seeded); the stored
 * log-prob is the un-tempered log_softmax entry; bookkeeping as sc_greedy_step. */
int sc_sample_step(const float* logits, int R, int V, int L, int t, int eos, int decoding_constraint, float temperature,
                   const float* uniforms, unsigned long long seed, int* seq, float* seq_lp, int* tokens, int* unfinished,
                   int* live_count, sc_stream_t stream);

/* K8 — state[i][:, state_ix] (models/caption_model.py:106-110): dst[r] = src[idx[r]], rows of row_bytes */
int sc_cache_reorder(const void* src, void* dst, const int* idx, long rows, long row_bytes, sc_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Training side (teacher forcing forward/backward, SURVEY.md rows a4, a5, a14; K2, K4/K9 backward, K10)
 * ------------------------------------------------------------------------------------------------------------ */

/* sc_linear with inverted dropout in the epilogue: y = dropout(act(x (W.m)^T + b), p) + residual
 * (nn.Dropout after the FFN ReLU / sublayer outputs / att_embed: models/transformer.py:325,356-358,
 * relation_transformer.py:327-329).  Dropout mask = Philox(drop_seed, drop_stream, element). */
int sc_linear_dropout(const void* x, int x_dtype, const void* w, int w_dtype, const float* mask, int mask_mode,
                      const float* uniforms, unsigned long long seed, unsigned long long stream_id, const float* bias,
                      const float* residual, void* y, int y_dtype, int M, int N, int K, int relu, int tile_n,
                      float dropout_p, unsigned long long drop_seed, unsigned long long drop_stream, sc_stream_t stream);

/* K2 — autograd of MaskedLinear (pruning/sampler.py:15-17,32-34): dWm[N,K] = dyT[N,M] * xT[K,M]^T with the fused
 * straight-through epilogue  dW (+)= dWm.m ;  dS (+)= dWm.W.sigmoid'(S) [.1 if bypass or raw] + sparsity_coeff*sigmoid'(S).
 * dyT/xT are transposed activations (M = padded token count, multiple of 8 for bf16).
 * workspace (optional, device, 16-byte aligned, >= N*K*4 bytes; more bytes allow more K splits): when given, the GEMM
 * stores split-K partial products there and a second kernel reduces them and applies the epilogue once per element
 * (measured faster than the fused epilogue for every shape of this model, DESIGN.md K2); NULL = single fused kernel. */
int sc_linear_wgrad(const void* dyT, const void* xT, int dtype, const float* w, const float* mask, int mask_mode,
                    const float* uniforms, unsigned long long seed, unsigned long long stream_id, int bypass_sigmoid_grad,
                    float sparsity_coeff, float* dw, float* ds, int accumulate, int N, int K, int M, int tile_n,
                    void* workspace, size_t workspace_bytes, sc_stream_t stream);

/* K2 without transposed operands (bf16): dy [M, N] and x [M, K] row-major, read as MN-major UMMA tiles through TMA boxes
 * of 64 tokens x 64 features; M needs no padding.  Two-kernel form, workspace as for sc_linear_wgrad (required). */
int sc_linear_wgrad_rowmajor(const void* dy, const void* x, const float* w, const float* mask, int mask_mode,
                             const float* uniforms, unsigned long long seed, unsigned long long stream_id,
                             int bypass_sigmoid_grad, float sparsity_coeff, float* dw, float* ds, int accumulate, int N, int K,
                             int M, void* workspace, size_t workspace_bytes, sc_stream_t stream);

/* out = g*keep*scale (cast), outT = its transpose (leading dim ldT, caller zero-pads); keep = (h != 0) when the saved
 * post-ReLU/dropout activation h is given, else the regenerated Philox dropout mask when dropout_p > 0.
 * colsum_accum (optional, fp32 [cols], pre-zeroed or holding a running sum): += column sums of `out` = the bias gradient. */
int sc_prep_grad(const float* g, const void* h, int h_dtype, void* out, void* outT, int ldT, int out_dtype, int rows, int cols,
                 float scale, float dropout_p, unsigned long long seed, unsigned long long stream_id, float* colsum_accum,
                 sc_stream_t stream);
int sc_transpose(const void* x, int x_dtype, void* y, int ldT, int y_dtype, int rows, int cols, sc_stream_t stream);
/* (W . mask)^T -> [K,N]: B operand of the dX GEMM; out_plain (optional, same dtype, [N,K]) receives W . mask from the
 * same pass, i.e. the forward operand and its transpose share one mask sample and one read of W and S */
int sc_apply_mask_transposed(const float* w, const float* mask, int mask_mode, const float* uniforms, unsigned long long seed,
                             unsigned long long stream_id, void* outT, int out_dtype, int N, int K, void* out_plain,
                             sc_stream_t stream);
/* every masked weight of a training step in one launch.  descs: device array of n_desc descriptors of ten 64-bit words
 * {w, s, uniforms, out [N,K], outT [K,N] (either may be 0), N, K (multiple of 4), stream_id, tile_start, tiles_k}; tensor i
 * owns the 64x64 tiles [tile_start_i, tile_start_{i+1}), tiles_k = ceil(K/64); element e of tensor i uses the Philox
 * stream stream_base + stream_id_i, i.e. the same sample sc_apply_mask_transposed / the wgrad epilogues regenerate
 * (replaces the per-layer sigmoid -> bernoulli -> mul chain of sparse_caption/pruning/masked_layer.py:84-110) */
int sc_apply_mask_batched(const void* descs, int n_desc, long total_tiles, int mask_mode, unsigned long long seed,
                          unsigned long long stream_base, int out_dtype, sc_stream_t stream);
/* elementwise straight-through gradient from a dense dWm (embedding table, WG heads) */
int sc_mask_grad(const float* dwm, const float* w, const float* mask, int mask_mode, const float* uniforms,
                 unsigned long long seed, unsigned long long stream_id, int bypass_sigmoid_grad, float sparsity_coeff,
                 float* dw, float* ds, int accumulate, size_t n, sc_stream_t stream);
int sc_colsum(const void* x, int dtype, float* out, int rows, int cols, int accumulate, sc_stream_t stream);

/* backward of the reference LayerNorm (models/transformer.py:329-341); dres (optional) is added to dx; da/db accumulate */
int sc_layernorm_bwd(const float* x, const float* a, const void* dy, int dy_dtype, const float* dres, float* dx, float* da,
                     float* db, int rows, int D, float eps, sc_stream_t stream);

/* dX GEMM of a linear whose input was h = dropout(relu(.)) (feed_forward.w_2, models/transformer.py:315-325): y bf16 [M,N] =
 * (x w^T) * scale where h (bf16 [M,N]) != 0, else 0 = the gradient operand of the previous linear; colsum (fp32 [N],
 * accumulated, may be NULL) += column sums of y = its bias gradient.  x bf16 [M,K], w bf16 [N,K]. */
int sc_linear_hmask(const void* x, const void* w, const void* h, float scale, float* colsum, void* y, int M, int N, int K,
                    sc_stream_t stream);

/* the same backward, also preparing the gradient operand of the NEXT linear of the backward chain (o-proj / ff2, whose
 * output gradient is dx): next_gb bf16 [rows, D] = dx (.) dropout keep mask of that linear's forward (Philox(seed,
 * stream_id, element), p = next_dropout_p), next_colsum fp32 [D] += its column sums (the bias gradient).  D == 512. */
int sc_layernorm_bwd_fused(const float* x, const float* a, const void* dy, int dy_dtype, const float* dres, float* dx, float* da,
                           float* db, int rows, int D, float eps, void* next_gb, float* next_colsum, float next_dropout_p,
                           unsigned long long seed, unsigned long long stream_id, sc_stream_t stream);

/* log_softmax (+ LanguageModelCriterion fwd/bwd when target != NULL): transformer.py:413, utils/losses.py:32-43 */
int sc_logsoftmax_nll(const float* logits, const int* target, const float* weight, const float* inv_norm, float* loss_sum,
                      void* dlogits, int d_dtype, float* logprobs, int rows, int V, sc_stream_t stream);
int sc_embedding_bwd(const int* tokens, const float* dy, float* dtable, int rows, int D, int V, float scale, sc_stream_t stream);

/* PruningMixin.compute_sparsity_loss from the binarized count (pruning/prune.py:228-269):
 * out3 = { |target - sparsity|, d(scaled loss)/d(nnz), sparsity } */
int sc_sparsity_coeff(const unsigned long long* count, double total, float target, float scale, const float* scale_dev,
                      float* out3, sc_stream_t stream);
/* clip_grad_value_ + Adam on a flat buffer (utils/optim.py:116-126,187-191); sigmoid_grad_coeff (device scalar, optional)
 * adds coeff*sigmoid'(param) to the gradient before clipping (sparsity loss on the mask-logit group).
 * CUDA-graph replay: values that change every step may live in device memory instead of the (baked) arguments -
 *   dyn (optional) = {lr, 1 - beta1^step, sqrt(1 - beta2^step)} overrides lr / step;  scale_dev overrides scale;
 *   every `seed` argument of this ABI with bit 63 set is a device pointer (low 63 bits) to the 64-bit seed. */
int sc_adam_clip(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr, float beta1, float beta2,
                 float eps, float weight_decay, float clip_value, float grad_scale, int step, const float* sigmoid_grad_coeff,
                 const float* dyn, sc_stream_t stream);

/* Whole-model optimizer step in one launch with the straight-through epilogue of the masked weights inside it: the flat
 * gradient buffer holds dWm = d loss / d (W . m) for masked tensors (what data-parallel ranks all-reduce - half the bytes of
 * dW + dS) and ordinary gradients for unmasked parameters.  Per masked element the step's mask sample is regenerated
 * (Philox(seed, stream_base + desc.stream, element) / uniforms / binarize / raw), dW = dWm * m, dS = dWm * W * sigmoid'(S)
 * [+ coeff * sigmoid'(S)] (pruning/sampler.py:10-34, prune.py:249-258), then clip + Adam for both parameter groups
 * (utils/optim.py:116-126,187-191; scripts/train_n_prune_transformer.py:67-82).
 * descs: device int64 [n_desc][5] = {w_off, s_off (-1 = unmasked), n, stream, first block}; one CTA per
 * sc_adam_clip_st_chunk() elements.  dyn (optional, device fp32) = {lr_w, 1 - b1^t, sqrt(1 - b2^t), lr_s}. */
int sc_adam_clip_st_chunk(void);
int sc_adam_clip_st(const void* descs, int n_desc, long total_blocks, float* w, const float* grad_wm, float* m_w, float* v_w, float* s,
                    float* m_s, float* v_s, const float* uniforms, int mask_mode, int bypass_sigmoid_grad, int update_logits,
                    unsigned long long seed, unsigned long long stream_base, float lr_w, float eps_w, float weight_decay_w, float lr_s,
                    float eps_s, float beta1, float beta2, float clip_value, float grad_scale, int step,
                    const float* sigmoid_grad_coeff, const float* dyn, sc_stream_t stream);

/* CIDEr-D reward of SCST on the device (scst/cider/pyciderevalcap/ciderD/ciderD_scorer.py:133-212 as used by
 * scst/scorers.py:47-114): one score per hypothesis (word ids [H, L], words = ids before the first <eos>, pads dropped) against
 * the references of image hyp_img[h].  n-grams (n <= 4, ids < 65536) are exact 64-bit keys (id_j << 16 j).
 * df_keys ascending with df_log = log(max(1, df)); ref_len = log(#documents); references of image b are
 * [img_ref_off[b], img_ref_off[b+1]), reference r owns n-gram entries [ref_ng_off[r], ref_ng_off[r+1]) of ref_keys (ascending)
 * / ref_vec (tf-idf), ref_norm [R,4], ref_length [R] (the scorer's bigram count).  Double precision, reference summation order. */
int sc_ciderd_score(const int* hyp, int H, int L, const int* hyp_img, int eos, int pad, const unsigned long long* df_keys,
                    const double* df_log, long n_df, double ref_len, double sigma, const long* img_ref_off, const long* ref_ng_off,
                    const unsigned long long* ref_keys, const double* ref_vec, const double* ref_norm, const int* ref_length,
                    double* out, sc_stream_t stream);
/* coco-caption validation metrics on word ids (coco_caption/eval.py:15-86 as called by eval_on_split, utils/training.py:257-327),
 * METEOR / SPICE / the PTB tokenizer excepted.  Hypotheses hyp int32 [H, L <= 64] (words = ids before the first <eos>, pads
 * dropped), each scored against the references of image hyp_img[h] in [0, n_images) and written to that image's slot;
 * hypotheses with an image index outside that range are skipped (sc_bleu_stats counts them in *bad_index).  References of image
 * b are [img_ref_off[b], img_ref_off[b+1]).
 * sc_cider_score: CIDEr of pycocoevalcap cider/cider_scorer.py (compute_cider: counts2vec + sim without the clip and the length
 * penalty of CIDEr-D); the tables are those of sc_ciderd_score, out float64 [n_images]. */
int sc_cider_score(const int* hyp, int H, int L, const int* hyp_img, int n_images, int eos, int pad, const unsigned long long* df_keys,
                   const double* df_log, long n_df, double ref_len, const long* img_ref_off, const long* ref_ng_off,
                   const unsigned long long* ref_keys, const double* ref_vec, const double* ref_norm, double* out, sc_stream_t stream);
/* BLEU sufficient statistics of bleu/bleu_scorer.py (cook_test, n = 4, option "closest"): stats int64 [n_images, 10] =
 * correct_1..4 (sum over n-grams of min(hypothesis count, largest count in one reference)), guess_1..4 = max(0, |h| - k + 1),
 * testlen = |h|, reflen = the reference length l minimising (|l - |h||, l).  Per image b: n-gram keys ascending in
 * keys[img_key_off[b] .. img_key_off[b+1]) with their max_count; reference r has length ref_tok_off[r+1] - ref_tok_off[r].
 * hyp_count[b] += 1 per hypothesis of image b. */
int sc_bleu_stats(const int* hyp, int H, int L, const int* hyp_img, int n_images, int eos, int pad, const long* img_key_off,
                  const unsigned long long* keys, const int* max_count, const long* img_ref_off, const long* ref_tok_off,
                  long long* stats, int* hyp_count, int* bad_index, sc_stream_t stream);
/* ROUGE-L of rouge/rouge.py (beta = 1.2) from the exact LCS with every reference (bit-parallel over the hypothesis positions):
 * out float64 [n_images].  Reference r's tokens are ref_tok[ref_tok_off[r] .. ref_tok_off[r+1]), any length. */
int sc_rouge_l(const int* hyp, int H, int L, const int* hyp_img, int n_images, int eos, int pad, const long* img_ref_off,
               const long* ref_tok_off, const int* ref_tok, double* out, sc_stream_t stream);
/* One launch, fixed order (bitwise reproducible): out float64 [9 + 6 n_images] = corpus Bleu_1..4 (bleu_scorer.py compute_score
 * on the summed statistics), mean ROUGE_L, mean CIDEr, #images without a hypothesis, #images with more than one, *bad_index;
 * then per image {Bleu_1..4 (compute_score's bleu_list), ROUGE_L, CIDEr} (coco-caption's imgToEval). */
int sc_caption_metrics_reduce(const long long* bleu_stats, const double* rouge, const double* cider, const int* hyp_count,
                              const int* bad_index, int n_images, double* out, sc_stream_t stream);
/* SCST rollout -> teacher-forcing inputs of the training step (utils/training.py:239-255 with RewardCriterion, utils/losses.py:10-29),
 * one launch.  seq int32 [R = B*S, L]: the rollout (S samples per image, rows image-major).  score float64 [R]: the samples'
 * CIDEr-D; base_score float64 [B] (the greedy baseline, one per image) or NULL (each sample's baseline is the mean of its image's
 * other S - 1 samples, S >= 2).  reward[r] = cider_weight * (score[r] - baseline[r]), rounded to fp32.  Writes [R, L]:
 * tokens = [bos, s_0 .. s_{L-2}], targets = s, key_valid = (tokens != pad), tok_w = reward * mask with mask[r, 0] = 1,
 * mask[r, t] = (s_{t-1} != pad); mask_sum (optional) = sum of mask; inv_norm = 1 / (norm_in ? *norm_in : sum of mask)
 * (norm_in: the data-parallel global count); mean_reward (optional) = mean of reward over the R rows. */
int sc_scst_targets(const int* seq, int R, int L, int S, const double* score, const double* base_score, float cider_weight,
                    int bos, int pad, int* tokens, int* targets, float* tok_w, float* key_valid, float* mask_sum, float* inv_norm,
                    const float* norm_in, float* mean_reward, sc_stream_t stream);

/* Magnitude / SNIP mask updates on flat buffers (PruningMixin.update_masks_once + compute_mask, pruning/prune.py:259-289 and the
 * gradual schedule :375-433 that calls it).  descs: device int64 [n_desc][6] = {src_off, dst_off, n, group, pos_base, first_block}:
 * segment i is one masked tensor, elements src[src_off + e] of the criterion source (weights, or the SNIP saliency) and
 * mask_out[dst_off + e], e < n; `group` its selection group, pos_base + e its 32-bit position in that group (the tie-break);
 * one CTA per sc_prune_chunk() elements, segment i owns CTAs [first_block_i, first_block_{i+1}).
 * sc_prune_stats: sums [n_desc][2] (double) = per segment {sum x, sum x^2}, x = src, or rint(sigmoid(src)) when binarize
 *   (the per-tensor counts of calculate_sparsities, prune.py:124-144); with center (optional, the sums of a first call) the second
 *   column is sum (x - mean)^2 (two-pass variance: exactly 0 for a constant tensor).  partials: double [total_blocks][2] scratch.
 *   Fixed summation order: bitwise reproducible.
 * sc_prune_select: criterion SC_PRUNE_ABS |w| (mag_blind / mag_uniform), SC_PRUNE_DIST |(w - mean) / std| with the segment's mean
 *   and population std from `sums` of the centred pass (mag_dist), SC_PRUNE_SNIP sal / (sum of the group's sal) from `sums` (snip), computed in fp32 on
 *   the fly.  Per group the first group_k[g] elements in (criterion, position) order get 0, every other element 1 (the complete
 *   mask is written: a weight pruned earlier can come back).  -0.0 sorts as +0.0, NaN above every number.  group_k (device int64
 *   [n_groups]) in [0, group size).  workspace: 16-byte aligned, n_groups * 1056 + n_desc * 8 bytes. */
#define SC_PRUNE_ABS 0
#define SC_PRUNE_DIST 1
#define SC_PRUNE_SNIP 2
int sc_prune_chunk(void);
int sc_prune_stats(const void* descs, int n_desc, long total_blocks, const float* src, int binarize, const double* center,
                   double* partials, double* sums, sc_stream_t stream);
int sc_prune_select(const void* descs, int n_desc, long total_blocks, int n_groups, const long long* group_k, int criterion,
                    const float* src, const double* sums, float* mask_out, void* workspace, size_t workspace_bytes,
                    sc_stream_t stream);

/* teacher-forcing attention with saved probabilities + backward (decoder self: causal_T = T; cross: groups = images with
 * S*T query rows; encoder box attention: additive bias): transformer.py:230-295, relation_transformer.py:258-293 */
int sc_attention_fwd(const void* q, const void* k, const void* v, int ldq, int ldk, int ldv, int dtype, const float* key_valid,
                     const float* bias, float* probs, void* out, int ldo, int G, int Tq, int Tk, int h, int dk, int causal_T,
                     float dropout_p, unsigned long long seed, unsigned long long stream_id, sc_stream_t stream);
int sc_attention_bwd(const void* q, const void* k, const void* v, int ldq, int ldk, int ldv, int dtype, const float* probs,
                     const float* d_out, int ldd, float* dq, float* dk_, float* dv, int ldgq, int ldgk, int ldgv, float* dbias,
                     int G, int Tq, int Tk, int h, int dk, float dropout_p, unsigned long long seed,
                     unsigned long long stream_id, sc_stream_t stream);
/* the same backward with the gradient preparation of the q / k / v projections that follow in the backward chain fused in
 * (bf16 operands, d_k = 64): dq / dk / dv leave as bf16, bq / bk / bv (fp32 [h * d_k], accumulated, all or none) receive
 * their column sums = the projections' bias gradients. */
int sc_attention_bwd_bf16out(const void* q, const void* k, const void* v, int ldq, int ldk, int ldv, const float* probs,
                             const float* d_out, int ldd, void* dq, void* dk_, void* dv, int ldgq, int ldgk, int ldgv, float* bq,
                             float* bk, float* bv, float* dbias, int G, int Tq, int Tk, int h, int dk, float dropout_p,
                             unsigned long long seed, unsigned long long stream_id, sc_stream_t stream);
/* log(max(relu(WG_h . emb(i,j) + b_h), 1e-6)) for all heads, and its gradient to WG (relation_transformer.py:179-183,196-256) */
int sc_box_bias_fwd(const float* boxes, const float* wg_w, const float* wg_b, float* bias, int B, int N, int h, int trig,
                    float wave_len, sc_stream_t stream);
int sc_box_bias_bwd(const float* boxes, const float* bias, const float* dbias, float* dwg_w, float* dwg_b, int B, int N, int h,
                    int trig, float wave_len, sc_stream_t stream);
/* BoxRelationalEmbedding itself (relation_transformer.py:196-256) for callers of the static method: emb fp32 [B,N,N,64]
 * (sin block, cos block) or [B,N,N,4] (the four log-deltas) when trig == 0. */
int sc_box_embedding(const float* boxes, float* emb, int B, int N, int trig, float wave_len, sc_stream_t stream);
/* out = log(max(x, lo)) (box_attention's additive term from the relu'd geometry weights, relation_transformer.py:283-286);
 * with dy != NULL: out = dy / x where x > lo, else 0 (its gradient). */
int sc_log_clamp(const float* x, const float* dy, float* out, size_t n, float lo, sc_stream_t stream);
/* backward of a plain log_softmax (OutputEmbedding, transformer.py:405-413): dx = dy - exp(logprobs) * rowsum(dy) */
int sc_logsoftmax_bwd(const float* logprobs, const float* dy, float* dx, int rows, int V, sc_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SC_B200_H */
