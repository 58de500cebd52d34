/*
 * libalm_b200 — C ABI of the B200-native AudioLM hot path.
 *
 * The reference (lucidrains/audiolm-pytorch) has no FFI / plugin registry: its hot path is reached
 * through Python classes that call torch library kernels.  This header is the boundary a maintainer
 * would bind instead (ctypes stub shown in INTEGRATION.md).  Each entry point names the reference
 * call it replaces (file:line under /root/reference/audiolm_pytorch/).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch allocates everything);
 *     the library allocates nothing, never synchronises, and launches on the given stream;
 *   - return value: ALM_OK (0) or a negative alm_status; details go to stderr;
 *   - bf16 tensors are raw uint16 storage (torch.bfloat16), "f32" is IEEE float, ids are int64;
 *   - all row-major; leading dimensions in ELEMENTS.
 */
#ifndef ALM_B200_H_
#define ALM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* alm_stream_t; /* == cudaStream_t */

typedef enum alm_status {
  ALM_OK = 0,
  ALM_ERR_ARG = -1,
  ALM_ERR_ALIGN = -2,
  ALM_ERR_CUDA = -3,
  ALM_ERR_UNSUPPORTED = -4
} alm_status;

/* ---- runtime ------------------------------------------------------------------------------ */
int alm_version(void);
const char* alm_status_string(int code);
unsigned long long alm_launch_count(void); /* kernels launched by this library since the last reset */
void alm_reset_launch_count(void);

/* ---- dense contractions (tcgen05 + TMA) ---------------------------------------------------- */
/*
 * C[b,m,n] (op)= alpha * sum_k A(b,m,k) * B(b,n,k)  [+ bias[n]]        bf16 x bf16 -> fp32 accumulate in TMEM
 *   a_mn = 0: A(m,k) = A[b*strideA + m*lda + k]   ("K-major", e.g. activations x[M,K])
 *   a_mn = 1: A(m,k) = A[b*strideA + k*lda + m]   ("MN-major", e.g. dy^T for weight gradients)
 *   b_mn likewise for B(n,k).   c_fp32: 0 -> bf16 output, 1 -> fp32 output.
 *   acc_mode: 0 overwrite, 1 C += (read-modify-write), 2 C += with fp32 atomics (required when split_k > 1).
 * Replaces every nn.Linear / einsum on the transformer path: audiolm_pytorch.py:255,259 (FFN),
 * :293-294,303 (q/kv/out projections), :621,798 (logit Linear), :972,979,1335,1350,1357 (grouped
 * logit einsums), and their autograd backward (dgrad: b_mn=1, wgrad: a_mn=b_mn=1).
 * Alignment: A/B base 16 B, lda/ldb/strides multiples of 8 elements.
 */
int alm_gemm_bf16(const void* A, int a_mn, int64_t lda, int64_t strideA, const void* B, int b_mn, int64_t ldb,
                  int64_t strideB, void* C, int c_fp32, int64_t ldc, int64_t strideC, int M, int N, int K, int batch,
                  float alpha, const float* bias, int acc_mode, int split_k, alm_stream_t stream);

/* ---- multi-query attention (tcgen05 + TMA, flash-style online softmax) ----------------------- */
/*
 * Token embeddings of the three transformers (audiolm_pytorch.py:686-699, 896-918, 1188-1223): every position is the
 * sum of up to two rows of a handful of fp32 parameter tables [rows_k, d] (start token, nn.Embedding rows, quantizer
 * embedding).  tables / grad_tables: HOST array of n_tables <= 8 device pointers (16-B aligned); src: device int32
 * [M, 2], each entry (table_id << 24) | row or -1.  gather: out [M, d] = sum of the rows.  scatter (its backward):
 * grad_tables[id][row] += dout[m] with 16-byte vector reductions (the caller zeroes the grad tables).
 */
int alm_embed_gather(const float* const* tables, int n_tables, const int32_t* src, float* out, int M, int d,
                     alm_stream_t stream);
int alm_embed_scatter(float* const* grad_tables, int n_tables, const int32_t* src, const float* dout, int M, int d,
                      alm_stream_t stream);
/*
 * Key-padding / forgetful-causal mask in the form the attention kernels read: uint8 [b, n_k] (non-zero = attend) ->
 * uint32 bits [b, 4 * ceil(n_k / 128)], bit i of word w = key 32 w + i.  One call per forward (all layers and the
 * backward share the result); a 128-key tile then costs every CTA one 16-byte load instead of 128 byte tests per row.
 */
int alm_pack_key_mask(const void* key_mask, void* bits, int b, int n_k, alm_stream_t stream);
/*
 * o[b,i,h*64:(h+1)*64] = softmax_j( q[b,i,h,:]·k[b,j,:] * scale, masked ) · v[b,j,:]
 *   one shared k/v head of width 64 (MQA); key_mask: PACKED bits from alm_pack_key_mask (attend = 1), optional;
 *   causal: query i sees keys j <= i + (n_k - n_q) (right-aligned, as needed by the KV cache).
 *   lse[b,h,i] (optional, row stride lse_stride >= n_q) = log2-domain log-sum-exp (log2 sum_j 2^(s_ij*scale*log2e)) of the masked scores for the backward.
 * Replaces Attend.forward / flash_attn (attend.py:69-146) as called by Attention.forward
 * (audiolm_pytorch.py:390).  Fully masked rows produce zeros (the reference's flash path yields NaN).
 * q rows stride ldq (q may be a column slice of a fused qkv buffer); k/v rows stride ldk/ldv, batch
 * strides k_bstride/v_bstride (elements).
 * bias (optional, fp32 [h, n_q, bias_rstride], shared by all batches): added to the scaled scores before the
 * masks, i.e. the `sim = sim + attn_bias` of the non-flash path (attend.py:122-124) fed by
 * RelativePositionBias / cross_attn_bias / pos_bias_mlp (audiolm_pytorch.py:202-242, 926-936, 1229-1298).
 * bias_rstride >= n_k and a multiple of 4; the backward accumulates d(bias) into dbias (same layout) with
 * atomic adds - zero it once per step, every layer / batch adds into it.
 */
int alm_mqa_attn_fwd(const void* q, int64_t ldq, const void* k, int64_t ldk, int64_t k_bstride, const void* v,
                     int64_t ldv, int64_t v_bstride, const void* key_mask, void* o, int64_t ldo, float* lse,
                     int64_t lse_stride, const float* bias, int64_t bias_hstride, int64_t bias_rstride, int b, int h,
                     int n_q, int n_k, int causal, float scale, alm_stream_t stream);

/*
 * Backward of alm_mqa_attn_fwd (two tcgen05 kernels: dK/dV per key block accumulating over all heads
 * in TMEM, then dQ per query block).  lse/delta are [b, h, n_q_pad] with n_q_pad a multiple of 128;
 * delta = rowsum(dO * O) from alm_attn_delta.  Autograd of attend.py:69-146.
 */
int alm_mqa_attn_bwd(const void* q, int64_t ldq, const void* k, int64_t ldk, int64_t k_bstride, const void* v,
                     int64_t ldv, int64_t v_bstride, const void* d_o, int64_t lddo, const void* key_mask,
                     const float* lse, const float* delta, int n_q_pad, void* dq, int64_t lddq, void* dk,
                     int64_t lddk, void* dv, int64_t lddv, const float* bias, float* dbias, int64_t bias_hstride,
                     int64_t bias_rstride, int b, int h, int n_q, int n_k, int causal, float scale,
                     alm_stream_t stream);
int alm_attn_delta(const void* o, int64_t ldo, const void* d_o, int64_t lddo, float* delta /* [b,h,stride] */,
                   int64_t delta_stride, int b, int h, int n, alm_stream_t stream);

/*
 * Dense attention bias from a learned table (HBM-bound gather, scatter-add backward):
 *   out[h, i, j] = idx[i*n_k + j] >= 0 ? table[idx * heads + h] : override_h[h]     (idx == -1: override)
 * out is fp32 [heads, n_q, ld] with ld >= n_k (pad columns are written as 0).  Replaces the `x[rel_pos]`
 * gather of RelativePositionBias.forward (audiolm_pytorch.py:225-242), the torch.where with cross_attn_bias
 * (:926-936) and the index-select + where with null_pos_bias of the fine transformer (:1278-1298).
 * The backward accumulates into dtable [rows, heads] / doverride [heads] (zeroed by the caller).
 */
int alm_bias_gather_fwd(const float* table, const int32_t* idx, const float* override_h, float* out, int heads,
                        int n_q, int n_k, int64_t ld, alm_stream_t stream);
int alm_bias_gather_bwd(const float* dbias, const int32_t* idx, float* dtable, float* doverride, int heads, int n_q,
                        int n_k, int64_t ld, alm_stream_t stream);

/*
 * Incremental decoding against a static KV cache (config C5).  The cache fill level is read from device memory
 * (`len`), so a whole decode step has constant launch parameters and can be replayed from one CUDA graph:
 *   alm_kv_append       k_cache[b, *len, :] = kv_new[b, 0:64];  v_cache[b, *len, :] = kv_new[b, 64:128]
 *   alm_mqa_attn_decode o[b, h*64:(h+1)*64] = softmax over keys j <= *len of (q[b,h,:]·k_cache[b,j,:]*scale) · v_cache
 * k_cache / v_cache: bf16 [b, max_len, 64] with batch stride cache_bstride (elements); key_mask (uint8 [b, >=max_len],
 * row stride mask_bstride, 1 = attend) optional.  splits > 1 slices the keys over that many CTAs per sequence
 * (flash-decoding) and merges the partial softmax states in a second launch.  Replaces the per-step torch.cat of the cache and the n_q = 1
 * attention of Attention.forward (audiolm_pytorch.py:363-365, 390) inside generate (:1406-1511, 1608-1740, 1896-2039).
 */
/* out[r, n] = sum_k x[r, k] W[n, k] (+ bias[n]) for rows <= 8 (a decode step's Linear layers: weight-read bound;
 * one warp per output column over all SMs).  W bf16 [N, ldw] with zero padding to a multiple of 8 columns. */
int alm_gemv_bf16(const void* x, int64_t ldx, const void* W, int64_t ldw, void* out, int c_fp32, int64_t ldo,
                  const float* bias, int rows, int N, int K, alm_stream_t stream);
int alm_kv_append(const void* kv_new, int64_t ld, void* k_cache, void* v_cache, int64_t cache_bstride,
                  const int32_t* len, int max_len, int b, alm_stream_t stream);
int alm_mqa_attn_decode(const void* q, int64_t ldq, const void* k_cache, const void* v_cache, int64_t cache_bstride,
                        const int32_t* len, int max_len, const void* key_mask, int64_t mask_bstride, void* o,
                        int64_t ldo, float* workspace /* [b, splits, h, 66] fp32 when splits > 1 */, int splits, int b,
                        int h, float scale, alm_stream_t stream);

/* ---- fused logit head + cross entropy (the [M, V] fp32 logits never reach HBM) --------------------------------
 * Replaces `logits = head(x)` + `F.cross_entropy(logits, labels, ignore_index=...)` of the three wrappers' loss paths
 * (audiolm_pytorch.py:621, 798, 965-983, 1325-1361 heads; :1561-1565, 1836-1854, 2119-2137 losses).
 *   alm_gemm_head_ce mode 1 : X [M, K] bf16 (row stride ldx) times W [V, K] bf16 (row stride ldw) (+ bias [V] fp32); the GEMM
 *       epilogue reduces every (row, n tile) to {max, sum 2^(t - max)} of t = logit * log2(e) -> part [M, tiles, 2]
 *       (tiles = alm_gemm_head_ce_tiles(V)) and writes logit[label] -> lab_logit [M] (rows whose label is never a column,
 *       e.g. ignore_index = -1, are left untouched)
 *   alm_ce_finish           : part, lab_logit -> lse [M] (natural log), loss_rows [M] = lse - logit[label] (0 when ignored)
 *   alm_gemm_head_ce mode 2 : recomputes the GEMM and writes d loss / d logits = (softmax - onehot) * (*scale_num / *scale_den)
 *       as bf16 [M, ldd] (zero rows where label == ignore_index; columns >= V are not written: pre-zero the padding). */
int alm_gemm_head_ce_tiles(int V);
int alm_gemm_head_ce(const void* X, int64_t ldx, const void* W, int64_t ldw, const float* bias, const int64_t* labels,
                     int64_t ignore_index, int mode, float* part, float* lab_logit, const float* lse,
                     const float* scale_num, const float* scale_den, void* dlogits, int64_t ldd, int M, int V, int K,
                     alm_stream_t stream);
int alm_ce_finish(const float* part, int tiles, const float* lab_logit, const int64_t* labels, int64_t ignore_index,
                  float* lse, float* loss_rows, int M, alm_stream_t stream);

/* One decode step of the WHOLE 4-stream hyper-connection stack (all layers: hyper-connection pre, q / kv projections,
 * value residual, cache append, attention over the static cache, out projection, feed-forward with GEGLU + LayerNorm,
 * final depth connection + LayerNorm) in ONE persistent cooperative kernel with device-wide barriers: what
 * Transformer.forward does for one new token under kv_cache (audiolm_pytorch.py:446-560 as driven by generate,
 * :1406-1511, 1608-1740, 1896-2039).  rows b <= 4.
 *   layer_table : device array [n_layers][24] of device pointers, per layer
 *       0..7   attention-branch hyper-connection: norm gamma [d], dynamic_alpha_fn [d,5], dynamic_beta_fn [d],
 *              static_alpha [4,5], static_beta [4], dynamic_alpha_scale [1], dynamic_beta_scale [1], branch LayerNorm gamma [d]
 *       8..15  the same eight for the feed-forward branch
 *       16, 18, 19, 20  bf16 operands REGROUPED per CTA (G = alm_decode_stack_grid() CTAs, pc = ceil(N / G)): row
 *              (c * pc + l) of the [G * pc, K] copy is row (c + l * G) of the [N, K] operand, zero rows past N; operands:
 *              [to_q ; to_kv] [h*64 + 128, d], to_out [d, h*64], W1 [2*pad8(inner), d] (value rows then gate rows, each
 *              block padded to pad8(inner)), W2 [d, pad8(inner)] (zero-padded columns).  17: unused.
 *       21     the inner LayerNorm gamma [inner] (fp32)
 *       22..23 k_cache, v_cache of the layer: bf16 [b, max_len, 64], batch stride cache_bstride
 *   x fp32 [b, d] (embedding of the new token), out bf16 [b, d]; *len is the cache fill level: the new token is written
 *   at position *len and *len is incremented by the kernel.  scratch: alm_decode_stack_scratch_bytes() bytes, 256-B
 *   aligned, owned by the caller; its first word pair is {barrier counter, sticky error flag (1 = a barrier timed out)}. */
int alm_decode_stack_grid(void);
int64_t alm_decode_stack_scratch_bytes(int b, int d, int heads, int inner);
int64_t alm_decode_stack_trace_offset(int b, int d, int heads, int inner); /* debugging: phase stamps of -DALM_DSTEP_TRACE builds */
int alm_decode_stack_step(const void* layer_table, int n_layers, const float* x, void* out, const float* final_gamma,
                          int32_t* len, int max_len, int64_t cache_bstride, const void* key_mask, int64_t mask_bstride,
                          void* scratch, int64_t scratch_bytes, int b, int d, int heads, int inner, int value_residual,
                          float scale, int grid_ctas /* = alm_decode_stack_grid() */, alm_stream_t stream);

/* ---- Hyper-Connections residual streams fused with the pre-LayerNorm (HBM-bound) ---------------- */
/*
 * Internal layout: residual streams R [M, S=4, d] bf16, M = batch*seq.  One call per branch does
 *   R      = R_in + beta_prev (x) Y          depth connection of the previous branch
 *            (or R_s = x_expand for all s: expand_streams, audiolm_pytorch.py:524)
 *   bin, R_out = width connection of this branch (dynamic+static alpha/beta, RMSNorm over channels)
 *   xn     = LayerNorm(bin) * ln_gamma       the branch's pre-norm (audiolm_pytorch.py:347, 254)
 * aux [M, 54] keeps the tanh activations, 1/|R_s|, the pre-activations z and the LN mean/rstd for the backward.
 * Replaces hyper_connections.HyperConnections.forward as used at audiolm_pytorch.py:446-454,
 * 528-547 (third-party; restated in oracle/third_party.py).  Only streams == 4 is built.
 */
int alm_hc_pre_fwd(const void* R_in, const void* Y, const float* beta_prev, const float* x_expand,
                   const float* gamma_hc, const float* dyn_alpha, const float* dyn_beta, const float* static_alpha,
                   const float* static_beta, const float* alpha_scale, const float* beta_scale,
                   const float* ln_gamma, void* R_out, void* bin, void* xn, float* beta_out, float* aux, int M,
                   int d, int streams, alm_stream_t stream);
int alm_hc_pre_bwd(const void* R_in, const void* Y, const float* beta_prev, const float* x_expand,
                   const float* gamma_hc, const float* dyn_alpha, const float* dyn_beta, const float* static_alpha,
                   const float* static_beta, const float* alpha_scale, const float* beta_scale,
                   const float* ln_gamma, const float* aux, const void* dR_out, const void* dxn,
                   const void* dbin_extra, const float* dbeta, void* dR_in, void* dY, float* dbeta_prev,
                   float* dx_expand, float dx_scale, float* g_gamma_hc, float* g_dyn_alpha, float* g_dyn_beta,
                   float* g_static_alpha, float* g_static_beta, float* g_alpha_scale, float* g_beta_scale,
                   float* g_ln_gamma, float* partial, int partial_blocks, int M, int d, int streams,
                   alm_stream_t stream);
/*
 * alm_hc_pre_bwd, d <= 1024: the per-channel parameter gradients are summed per CTA in fp32 into `partial`
 * (room for partial_blocks * (8*d + 32) floats; the kernel runs at most partial_blocks CTAs) and reduced from there
 * in a fixed order, so every parameter gradient is bitwise reproducible.  d > 1024 ignores `partial`.
 */
/* last depth connection + reduce_streams (sum) + final LayerNorm (audiolm_pytorch.py:551-555) */
int alm_hc_post_fwd(const void* R_in, const void* Y, const float* beta_prev, const float* ln_gamma, void* out,
                    float* stats, int M, int d, int streams, alm_stream_t stream);
int alm_hc_post_bwd(const void* R_in, const void* Y, const float* beta_prev, const float* ln_gamma,
                    const float* stats, const void* dout, void* dR_in, void* dY, float* dbeta_prev,
                    float* g_ln_gamma, int M, int d, int streams, alm_stream_t stream);

/* ---- plain residual + pre-LayerNorm (num_residual_streams == 1: Residual(branch), audiolm_pytorch.py:446) ------ */
/* r_new = r (+ y);  xn = LN(r_new) * gamma;  rb = bf16 copy of r_new (k/v projection input).  fp32 residual stream. */
int alm_resid_ln_fwd(const float* r, const void* y, const float* gamma, float* r_new, void* xn, void* rb, float* stats,
                     int M, int d, alm_stream_t stream);
/* dr = out_scale * (dr_out + LayerNorm-backward(dxn) + dextra);  g_gamma += dxn * xhat */
int alm_resid_ln_bwd(const float* r_new, const float* gamma, const float* stats, const float* dr_out, const void* dxn,
                     const void* dextra, float* dr, void* dr_bf16, float* g_gamma, float out_scale, int M, int d,
                     alm_stream_t stream);

/* ---- FeedForward inner part: GEGLU + LayerNorm(inner) (audiolm_pytorch.py:246-258) -------------- */
/* h [M, ldh] bf16 holds a = h[:, 0:inner] and gate = h[:, gate_off:gate_off+inner];
 * gn[M, ldg] = LN(gelu(gate) * a) * gamma, columns [inner, inner_pad) are written as zeros. */
int alm_geglu_ln_fwd(const void* h, int64_t ldh, int gate_off, const float* gamma, void* gn, int64_t ldg,
                     float* stats, int M, int inner, int inner_pad, alm_stream_t stream);
int alm_geglu_ln_bwd(const void* h, int64_t ldh, int gate_off, const float* gamma, const float* stats,
                     const void* dgn, int64_t ldg, void* dh, float* g_gamma, int M, int inner, int inner_pad,
                     alm_stream_t stream);

/* ---- cross entropy with ignore_index, fused forward + d(logits) --------------------------------- */
/* loss_rows[r] = lse(logits[r]) - logits[r, label]  (0 if label == ignore_index);
 * dlogits[r, 0:Vpad] (bf16, optional) = (softmax - onehot) * (*scale_num / *scale_den).
 * Replaces F.cross_entropy at audiolm_pytorch.py:1561-1565, 1839-1849, 2122-2132. */
int alm_ce_fwd_bwd(const float* logits, int64_t ldl, const int64_t* labels, int64_t ignore_index, float* loss_rows,
                   void* dlogits, int64_t ldd, const float* scale_num, const float* scale_den, int rows, int V,
                   int Vpad, alm_stream_t stream);

/* ---- sampling: top-k filter + Gumbel-max in one launch ------------------------------------------- */
/* ids[r] = argmax_c over the k largest logits of row r of (logits/temperature - log(-log(u+1e-20)+1e-20));
 * `uniform` is drawn by the caller (torch `uniform_`, same generator order as the reference) so sampled ids
 * are reproducible.  Replaces top_k + gumbel_sample (audiolm_pytorch.py:98-117) in the generate loops. */
int alm_topk_gumbel_sample(const float* logits, int64_t ldl, const float* uniform, int64_t ldu, int64_t* ids, int rows,
                           int V, int k, float temperature, alm_stream_t stream);

/* ---- small helpers on the same path ------------------------------------------------------------- */
/* out = alpha*x + beta*y (bf16, 2-D strided): value-residual mix v = 0.5 (v + v_first), :355-358 */
int alm_axpby_bf16(const void* x, int64_t ldx, float alpha, const void* y, int64_t ldy, float beta, void* out,
                   int64_t ldout, int64_t rows, int cols, alm_stream_t stream);
/* fp32 master weights -> zero-padded bf16 GEMM operands (what autocast does at every Linear) */
int alm_cast_pad_bf16(const float* src, int64_t lds, void* dst, int64_t ldd, int64_t rows, int cols, int cols_pad,
                      alm_stream_t stream);
/*
 * The same cast for MANY tensors in one launch (every Linear of a model after an optimizer step; what bf16 autocast does
 * per Linear per forward): desc_dev = device int64 [n][7] = {src ptr, dst ptr, rows, cols, cols_pad (even), lds, ldd}.
 */
int alm_cast_pad_multi(const int64_t* desc_dev, int n, alm_stream_t stream);
int alm_scale_by_scalar_bf16(void* x, const float* s, int64_t n, alm_stream_t stream);

/* ---- SoundStream codec (fp32) ---------------------------------------------------------------- */
/*
 * CausalConv1d (soundstream.py:332-345): left pad = dilation*(K-1) + 1 - stride filled in-kernel
 * (pad_mode 0 reflect [edge sample excluded], 1 zeros, 2 replicate), then conv with stride/dilation:
 *   y[b,o,t] = act( bias[o] + sum_c sum_j w[o,c,j] * xpad[b,c,t*stride + j*dilation] ) (+ residual[b,o,t])
 * act_elu = 1 applies ELU(alpha=1) before the residual add, which fuses a ResidualUnit
 * (soundstream.py:362-369) into two launches: conv_k7(dil)+ELU, then conv_k1+ELU+skip.
 * x [B,Cin,T], w [Cout,Cin,K], y [B,Cout,T/stride], all contiguous fp32.
 * w_packed = 1: w is the pre-transposed copy [Cin,K,Cout] (coalesced weight staging of the register-tiled
 * kernel; only for the (K, stride, dilation) shapes SoundStream uses: (7,1,{1,3,9}), (1,1,1), (3,1,1), (2s,s,1)
 * for s in 2,3,4,5,8 - other shapes take the generic kernel and need the torch layout).
 */
int alm_causal_conv1d_fwd(const float* x, const float* w, const float* bias, const float* residual, float* y, int B,
                          int Cin, int Cout, int T, int K, int stride, int dilation, int pad_mode, int act_elu,
                          int w_packed, alm_stream_t stream);
/* CausalConvTranspose1d (soundstream.py:347-360): kernel 2*stride, output trimmed to n*stride;
 * x [B,Cin,n], w [Cin,Cout,2*stride], y [B,Cout,n*stride]; polyphase form, 2 taps per input channel. */
/*
 * Fused ResidualUnit (soundstream.py:362-369): y = x + ELU(b1 + W1 . ELU(b7 + conv_k7,dilation(x))), causal padding
 * as above.  One launch; the k=7 result stays in shared memory.  Weights in the packed layout ([Cin,7,Cout] and
 * [Cin,1,Cout]); C in {32, 64, 128, 256}, dilation in {1, 3, 9} (else ALM_ERR_UNSUPPORTED: use the two conv calls).
 * Bit-identical to alm_causal_conv1d_fwd(k7, ELU) followed by alm_causal_conv1d_fwd(k1, ELU, residual).
 */
int alm_residual_unit_fwd(const float* x, const float* w7_packed, const float* b7, const float* w1_packed,
                          const float* b1, float* y, int B, int C, int T, int dilation, int pad_mode,
                          alm_stream_t stream);
/*
 * SoundStream encoder on the tensor cores (csrc/codec_tc.cu): split-bf16 ("bf16x3": x_hi w_hi + x_lo w_hi + x_hi w_lo,
 * fp32 accumulation) implicit-GEMM causal convs.  Activations travel between these three calls in the "C8S" layout
 *   bf16 [B][2C/8][P][T/P][8]   (chunk c < C/8: hi halves of channels 8c..8c+7, chunk C/8 + c: their lo halves;
 *                                P phase planes: time t lives in plane t % P, row t / P; same bytes as fp32 [B][C][T]).
 * Replaces the same reference calls as alm_causal_conv1d_fwd / alm_residual_unit_fwd (soundstream.py:332-383) when the
 * whole encoder runs in this format; results agree with the fp32 path to ~1e-5 relative.
 *
 * alm_codec_first_conv: CausalConv1d(1, Cout, K <= 8) on fp32 wave [B][T] -> C8S (P = 1).  Cout in {32, 64}.
 * alm_codec_ru_tc:      fused ResidualUnit  y = x + ELU(W1 ELU(W7 *_dil x + b7) + b1), C in {32, 64, 128, 256},
 *                       dilation <= 9; x in C8S (P = 1), y in C8S with out_phases planes.  w_units: bf16
 *                       [8 taps (7 = the 1x1 conv)][C/16 k-steps][hi, lo][2][C][8] (ops.pack_ru_weights).
 * alm_codec_conv_tc:    CausalConv1d(Cin, Cout, K, stride) with dilation 1; x in C8S with P = stride planes; y in C8S
 *                       (out_phases) or, out_fp32 = 1, fp32 channels-last [B][Tin/stride][Cout] (the RVQ input).
 *                       w_units: bf16 [Cout/BN][K][Cin/16][hi, lo][2][BN][8], BN = min(256, largest of 64/128/256 <= Cout).
 * pad_mode: 0 reflect, 1 constant zero, 2 replicate.
 */
int alm_codec_first_conv(const float* x, const float* w, const float* bias, void* y, int B, int T, int Cout, int K,
                         int pad_mode, alm_stream_t stream);
int alm_codec_ru_tc(const void* x, void* y, const void* w_units, const float* b7, const float* b1, int B, int C, int T,
                    int dilation, int pad_mode, int out_phases, alm_stream_t stream);
int alm_codec_conv_tc(const void* x, void* y, const void* w_units, const float* bias, int B, int Cin, int Cout, int Tin,
                      int K, int stride, int pad_mode, int out_phases, int out_fp32, int upsample, alm_stream_t stream);
/*
 * Decoder side (soundstream.py:347-360, 615-627).  CausalConvTranspose1d(Cin, C', 2s, stride s) runs as
 * alm_codec_conv_tc with K = 2, stride 1, constant padding, Cout = s * C' (ops.pack_convT_weights) and upsample = s:
 * output column block r of row t is written as time step t * s + r of a C8S tensor with C' channels.
 * alm_codec_pack_c8s: fp32 channels-last [B][n][C] (quantizer output) -> C8S (P = 1).
 * alm_codec_last_conv: CausalConv1d(Cin in {32, 64}, 1, K <= 8) on C8S -> fp32 wave [B][T].
 */
int alm_codec_pack_c8s(const float* x, void* y, int B, int n, int C, alm_stream_t stream);
int alm_codec_last_conv(const void* x, const float* w, const float* bias, float* y, int B, int T, int Cin, int K,
                        int pad_mode, alm_stream_t stream);
int alm_causal_convT1d_fwd(const float* x, const float* w, const float* bias, float* y, int B, int Cin, int Cout,
                           int n, int stride, alm_stream_t stream);
/*
 * Residual VQ, eval path (vector-quantize-pytorch ResidualVQ.forward as called at soundstream.py:840):
 * for q in 0..Q-1: idx = argmin_c sqrt(max(|r|^2 + |e_c|^2 - 2 r.e_c, 0)) (lowest index on ties);
 * r -= e_idx; quantized += e_idx.  x [N, D] (row stride ldx), codebooks [Q, C, D], indices [N, Q] int64.
 * e2_workspace: Q*C floats of scratch.
 */
int alm_rvq_encode(const float* x, int64_t ldx, const float* codebooks, float* e2_workspace, float* quantized,
                   int64_t ldq, int64_t* indices, int64_t ldi, int N, int D, int C, int Q, alm_stream_t stream);
/*
 * Residual VQ search with the distance GEMM on the tensor cores (csrc/rvq_tc.cu); same reference call as
 * alm_rvq_encode (soundstream.py:840).  Per stage q the host runs
 *     alm_gemm_bf16(R' [N, 3D], B'_q [C, 3D]) -> scores [N, C] fp32      (R' = [r_hi | r_lo | r_hi], B' = [e_hi | e_hi | e_lo])
 *     alm_rvq_select(scores, e2_q, codebook_q, r, quantized, R', indices + q, ...)
 * select re-evaluates every candidate within the bf16x3 error bound of the best approximate score with the exact fp32
 * expansion sqrt(max(|r|^2 + |e|^2 - 2 r.e, 0)) (lowest index on ties), then r -= e, quantized += e, R' <- split(r).
 * alm_rvq_pack_codebooks: codebooks fp32 [rows = Q*C, D] -> packed bf16 [rows, 3D] + e2 [rows] (once per weight version).
 * alm_rvq_prepare: r = x, quantized = 0, R' = split(x).
 */
int alm_rvq_pack_codebooks(const float* codebooks, void* packed, float* e2, int64_t rows, int D, alm_stream_t stream);
int alm_rvq_prepare(const float* x, int64_t ldx, float* r, float* quantized, int64_t ldq, void* rp, int N, int D,
                    alm_stream_t stream);
int alm_rvq_select(const float* scores, int64_t lds, const float* e2, const float* codebook, float* r, float* quantized,
                   int64_t ldq, void* rp, int64_t* indices, int64_t ldi, int N, int D, int C, int write_rp,
                   alm_stream_t stream);

/* get_output_from_indices (soundstream.py:697): out[n,:] = sum_q codebooks[q][indices[n,q]] (-1 -> skip) */
int alm_rvq_decode(const int64_t* indices, int64_t ldi, const float* codebooks, float* out, int64_t ldo, int N, int D,
                   int C, int Q, alm_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* ALM_B200_H_ */
