/* liblasr -- C ABI of the B200-native (sm_100a) kernels behind LiteASR's U2 + hybrid-CTC hot path.
 *
 * The reference (Nazukixv/LiteASR) has NO FFI: every FLOP on its hot path is a stock torch op
 * (SURVEY.md section 2.1).  Each entry point below therefore names the reference *call site* whose
 * arithmetic it replaces (paths relative to /root/reference/liteasr).  INTEGRATION.md shows the
 * ctypes binding a reference maintainer would add.
 *
 * Conventions
 *   - plain C: raw device pointers + sizes, no torch types; the caller (PyTorch) owns every buffer,
 *     the library never allocates or frees device memory and keeps no mutable global state
 *     (except the thread-local last-error string and a cached driver entry point).
 *   - every function enqueues on `stream` (a cudaStream_t passed as void*) and never synchronises;
 *     all of them are CUDA-graph capturable.
 *   - return 0 on success, a negative LASR_ERR_* on failure; lasr_last_error() describes it.
 *     Nothing throws across the ABI, nothing exits.  There is no CPU fallback.
 *   - dtype codes: LASR_F32 / LASR_BF16.  Math and accumulation are always fp32.
 */
#ifndef LASR_H
#define LASR_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LASR_OK 0
#define LASR_ERR_BAD_ARG (-1)
#define LASR_ERR_UNSUPPORTED (-2)
#define LASR_ERR_CUDA (-3)
#define LASR_ERR_DRIVER (-4)

#define LASR_F32 0
#define LASR_BF16 1

#define LASR_ACT_NONE 0
#define LASR_ACT_RELU 1
#define LASR_ACT_SWISH 2
#define LASR_ACT_MUL 3 /* only with `dact`: the saved tensor IS the factor (C = alpha * (A.B^T) * dact), see aux_deriv */

int lasr_version(void);             /* 100 * major + minor */
int lasr_arch(void);                /* 100 (sm_100a) */
const char* lasr_last_error(void);  /* thread-local, valid until the next failing call */
unsigned long long lasr_launch_count(void); /* kernels launched by this library so far (bench bookkeeping) */

/* ------------------------------------------------------------------------------------------------
 * GEMM  C[b1,b2] = alpha * act(A[b1,b2] . B[b1,b2]^T + bias) (+ res)
 *   bf16 operands -> tcgen05.mma (TMEM accumulators, TMA-fed, 128xBNx64 tiles);
 *   fp32 operands -> SIMT fp32 FMA kernel (the "fp32 parity mode").
 * Replaces every nn.Linear / 1x1 Conv1d / torch.matmul on the path:
 *   nets/feed_forward.py:18-19, nets/attention.py:35-37,56,58,132,145,149,
 *   nets/conformer_convolution.py:48,55, nets/subsampling.py:34,47 (via im2col),
 *   nets/ctc.py:29, nets/transformer_decoder.py:91 and their autograd backward GEMMs.
 *   trans_a = 0: A is (M,K) row-major with row stride lda;  1: A is stored (K,M) row-major.
 *   trans_b = 0: B is (N,K) row-major (nn.Linear weight);   1: B is stored (K,N) row-major.
 *   Two-level batching (b1 outer, b2 inner) with independent element strides, so head-interleaved
 *   (B,T,H,dk) tensors are addressed in place (stride 0 broadcasts an operand).
 *   aux (optional, C dtype/ldc): receives the pre-activation value (acc + bias).
 *   accumulate = 1: C (fp32) += alpha * A.B^T with red.global.add (split-K and batch-reduce wgrads);
 *                   bias/act/res/aux/dact/colsum must be unset; a C batch stride of 0 reduces over that batch level.
 * ------------------------------------------------------------------------------------------------ */
typedef struct lasr_gemm_args {
    const void* a;
    const void* b;
    void* c;
    const float* bias; /* [N] fp32 or NULL */
    const float* res;  /* fp32 residual, addressed like C (ldres) or NULL */
    void* aux;         /* optional pre-activation output (C dtype, ldc) */
    int32_t m, n, k;
    int32_t ab_dtype, c_dtype;
    int32_t trans_a, trans_b;
    int64_t lda, ldb, ldc, ldres;
    int32_t batch1, batch2;
    int64_t sa1, sa2, sb1, sb2, sc1, sc2; /* element strides per batch level (res/aux follow C) */
    float alpha;
    int32_t act;
    int32_t accumulate;
    int32_t split_k; /* >= 1; > 1 requires accumulate */
    /* backward-fusion extras (all optional):
     *   dact  : saved tensor of the forward activation (operand dtype, addressed like C with row stride lddact):
     *           C = alpha * (A.B^T) * act'(dact), act' = swish'(pre-activation) | relu'(activation output);
     *           replaces the separate activation-backward pass of nets/feed_forward.py:18-19; no bias/res/aux.
     *   colsum: fp32 vector, colsum[b1*cs1 + b2*cs2 + n] += sum_m C[m,n] (red.add): the bias gradient of the
     *           nn.Linear that produced this GEMM's A-side gradient, without re-reading C. */
    const void* dact;
    int64_t lddact;
    float* colsum;
    int64_t cs1, cs2;
    /* n_store: 0, or n <= n_store <= ldc: columns [n, n_store) of C are also written (with zeros: B has no such rows).
     * Lets a ragged N (T' = 299 attention scores in a 304-wide buffer) run entirely on the vector epilogue; the consumer
     * ignores those padding columns.  No bias/res/aux/dact/colsum. */
    int32_t n_store;
    /* dropout on the output (optional; the reference's nn.Dropout sites that sit right behind a Linear: nets/feed_forward.py:19,
     * nets/conformer_layer.py:42,54,63,125, nets/transformer_layer.py:48,58,174, nets/positional_encoding.py:75, and -- as the
     * backward of nets/ctc.py:29 -- the input gradient of ctc_lo):
     *   C = keep(m,n) * drop_scale * alpha * act(A.B^T + bias)  (+ res: the residual is added AFTER the mask)
     * keep(m,n) comes from Philox4x32-7 keyed by drop_state = device {seed, step} (two uint64), drop_site and the element's
     * (row, column) -- see the "dropout" section below; drop_thr = round(p * 32768) <= 0x7c00 (0 = off), drop_scale = 32768 / (32768 - thr).
     * drop_mark_aux = 1: dropped elements of `aux` (the saved pre-activation) receive -1e30, whose act'() is exactly 0, so the
     * activation-backward GEMM (dact = aux) applies the SAME mask without regenerating it (its alpha carries drop_scale).
     * Unbatched GEMMs only; not with accumulate / dact / n_store. */
    const void* drop_state;
    uint32_t drop_site;
    uint32_t drop_thr;
    float drop_scale;
    int32_t drop_mark_aux;
    /* aux_deriv = 1 (act = swish, aux set): `aux` receives act'(A.B^T + bias) -- the DERIVATIVE of the activation at the
     * pre-activation -- instead of the pre-activation itself, and 0 at elements dropped by drop_mark_aux.  The backward GEMM then
     * runs with dact = aux, act = LASR_ACT_MUL: one multiply per element instead of re-evaluating swish'() (tanh + 6 flops) in an
     * epilogue that is instruction-bound (nets/feed_forward.py:18-19 backward), and lasr_ffn_bwd consumes the same tensor. */
    int32_t aux_deriv;
} lasr_gemm_args;

int lasr_gemm(const lasr_gemm_args* args, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Weight gradient of a Linear on CTA pairs (tcgen05.mma.cta_group::2):  c (M, N fp32, row stride ldc) += alpha * a^T . b with
 * a (K, M) and b (K, N) row-major bf16 -- dW += dy^T x, the autograd backward of every nn.Linear of the path (nets/feed_forward.py:
 * 18-19, nets/attention.py:35-37, nets/conformer_convolution.py:48,55).  Same contract as lasr_gemm(trans_a = trans_b = 1,
 * accumulate = 1, split_k); needs M % 256 == 0 and N % 256 == 0 (lasr_wgrad2_supported): each CTA of a pair stages only its half of
 * both operands for a 256 x 256 tile.
 * ------------------------------------------------------------------------------------------------ */
int lasr_wgrad2_supported(int m, int n);
int lasr_wgrad2(const void* a, int64_t lda, const void* b, int64_t ldb, float* c, int64_t ldc, float alpha, int m, int n, int k, int split_k,
                void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused backward of the two inner GEMMs of a position-wise feed-forward block (nets/feed_forward.py:18-19 backward; the
 * encoder runs the block twice per Conformer layer, nets/conformer_layer.py:37-47,58-66), bf16 / tcgen05:
 *     dh  (M, f) = alpha * (dy (M, d) . W2 (d, f)) * g (M, f)      W2 = fc2.weight, g = act'(fc1 pre-activation) saved by the
 *                                                                 forward GEMM (aux_deriv; 0 where the inner dropout dropped)
 *     colsum (f) += sum_rows dh                                    fc1's bias gradient (optional)
 *     dln (M, d) = dh . W1 (f, d)                                  W1 = fc1.weight
 * One persistent kernel: a 128-row tile of dh exists only as 64-column chunks that go TMEM -> registers -> a shared-memory slab
 * that is both the A operand of the second MMA and the source of the bulk tensor store of dh (kept for the fc1 weight-gradient
 * GEMM).  Replaces lasr_gemm(dact) + lasr_gemm for d % 64 == 0, 64 <= d <= 256, f % 64 == 0 (lasr_ffn_bwd_supported); other
 * shapes return LASR_ERR_UNSUPPORTED.  All matrices row-major with 16-byte aligned bases and row strides.
 * ------------------------------------------------------------------------------------------------ */
int lasr_ffn_bwd_supported(int d, int f);
void lasr_ffn_bwd_set_trace(void* buf); /* developer aid: 32 x 8 clock64 stamps of CTA 0's first chunks (NULL = off) */
int lasr_ffn_bwd(const void* dy, int64_t lddy, const void* g, int64_t ldg, const void* w2, int64_t ldw2, const void* w1, int64_t ldw1,
                 void* dh, int64_t lddh, void* dln, int64_t lddln, float* colsum, float alpha, int M, int d, int f, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused FORWARD of the same block (nets/feed_forward.py:18-19 with the Swish activation, inside nets/conformer_layer.py:37-47
 * and :58-66: x + ff_scale * dropout(ff(LN x))), bf16 / tcgen05, one persistent kernel:
 *     a   (M, f) = drop_in(swish(ln (M, d) . W1 (f, d)^T + b1))         bf16, kept for fc2's weight gradient
 *     g   (M, f) = swish'(ln . W1^T + b1), 0 where drop_in dropped       bf16, what lasr_ffn_bwd multiplies by
 *     out (M, d) = res + drop_out(alpha * (a . W2 (d, f)^T + b2))         fp32 residual stream (res fp32, may alias nothing)
 * The pre-activation never exists in memory and a is not read back: a 128-row tile of a lives as 64-column chunks that go
 * TMEM -> registers -> a shared-memory slab that is the A operand of the second MMA and the source of its bulk tensor store.
 * Replaces lasr_gemm(act = Swish, aux_deriv) + lasr_gemm(res) for the shapes of lasr_ffn_fwd_supported (= lasr_ffn_bwd's).
 * Dropout: the two sites share drop_state; *_thr = 0 switches a site off (see "Dropout" below).
 * ------------------------------------------------------------------------------------------------ */
int lasr_ffn_fwd_supported(int d, int f);
int lasr_ffn_fwd(const void* ln, int64_t ldln, const void* w1, int64_t ldw1, const float* b1, const void* w2, int64_t ldw2, const float* b2,
                 const float* res, int64_t ldres, void* a, int64_t lda, void* g, int64_t ldg, float* out, int64_t ldout, float alpha, int M, int d,
                 int f, const void* drop_state, uint32_t in_site, uint32_t in_thr, float in_scale, uint32_t out_site, uint32_t out_thr,
                 float out_scale, void* stream);

/* ------------------------------------------------------------------------------------------------
 * CTC forward-backward fused with the log-softmax backward.
 * Replaces criterions/hybrid_ctc_attn.py:67-75 (transpose + log_softmax + nn.CTCLoss(sum) and the
 * autograd backward of all three).  logits (T,B,V) with element strides (st, sb, 1) so the model's
 * (B,T',V) tensor is consumed in place; targets (B,lmax) int64 padded (any value) beyond tgt_len.
 *   nll[b]          = -log p(l_b | x_b)   (+inf when infeasible, like zero_infinity=False)
 *   grad[t,b,c]     = grad_scale * upstream * (softmax[t,b,c] - occupancy[t,b,c])  for t <  in_len[b]
 *                   = 0                                                            for t >= in_len[b]
 *   upstream: optional device scalar (fp32) multiplied into grad_scale (autograd's grad_output).
 * Workspace: lasr_ctc_workspace_bytes(T,B,lmax).
 * ------------------------------------------------------------------------------------------------ */
size_t lasr_ctc_workspace_bytes(int T, int B, int lmax);
int lasr_ctc_fwdbwd(const void* logits, int dtype, int64_t st, int64_t sb, const int64_t* targets,
                    const int64_t* in_len, const int64_t* tgt_len, int T, int B, int V, int lmax, int blank,
                    float grad_scale, const float* upstream, float* nll, void* grad, int64_t gst, int64_t gsb,
                    void* workspace, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * LayerNorm over the last dim (nets/layer_norm.py:8-29, eps 1e-12) and its backward.
 *   fwd: y = (x - mean) * rstd * gamma + beta; x fp32 (rows,d) row stride ldx; y fp32|bf16.
 *   bwd: dx (+)= LN'(dy) (accumulate = 1 adds into dx: the residual-stream gradient);
 *        dgamma/dbeta are ACCUMULATED (red.add) into the caller's (pre-zeroed) gradient buffers.
 *        Optional fused outputs (NULL to skip): dx_lo = bf16 copy of the final dx (operand of the next block's
 *        backward GEMMs); colsum[d] += colsum_scale * sum_rows dx (bias gradient of the Linear feeding this residual).
 * d % 4 == 0, d <= 1024; dgamma/dbeta/colsum 16-byte aligned.
 * ------------------------------------------------------------------------------------------------ */
int lasr_layernorm_fwd(const float* x, int64_t ldx, const float* gamma, const float* beta, void* y, int y_dtype,
                       int64_t ldy, float* mean, float* rstd, int rows, int d, float eps, void* stream);
int lasr_layernorm_bwd(const void* dy, int dy_dtype, int64_t lddy, const float* x, int64_t ldx, const float* mean,
                       const float* rstd, const float* gamma, float* dx, int64_t lddx, int accumulate, float* dgamma,
                       float* dbeta, int rows, int d, void* dx_lo, int64_t lddxlo, float* colsum, float colsum_scale,
                       void* stream);
/* The same with (a) dx_lo of either dtype (lo_dtype = LASR_BF16 | LASR_F32) and (b) dropout applied to the two fused outputs:
 * the block that consumes dx_lo / colsum sits behind nn.Dropout on its output in the forward pass (x + drop(f(LN x)),
 * nets/conformer_layer.py:37-66, nets/transformer_layer.py:29-61,161-177), so what it must receive is keep * scale * dx with
 * the mask of THAT site, regenerated here; dx itself stays unmasked.  drop_thr = 0: identical to lasr_layernorm_bwd. */
int lasr_layernorm_bwd_drop(const void* dy, int dy_dtype, int64_t lddy, const float* x, int64_t ldx, const float* mean,
                            const float* rstd, const float* gamma, float* dx, int64_t lddx, int accumulate, float* dgamma,
                            float* dbeta, int rows, int d, void* dx_lo, int lo_dtype, int64_t lddxlo, float* colsum,
                            float colsum_scale, const void* drop_state, uint32_t drop_site, uint32_t drop_thr, float drop_scale,
                            void* stream);

/* ------------------------------------------------------------------------------------------------
 * Dropout (the reference's nn.Dropout / F.dropout sites: nets/positional_encoding.py:55,75, nets/attention.py:55,
 * nets/feed_forward.py:19, nets/conformer_layer.py:42,54,63,125, nets/transformer_layer.py:48,58,174, nets/ctc.py:29).
 * torch's generator stream cannot be replayed by fused kernels, so the masks come from the library's own counter-based
 * stream (Philox4x32 with 7 rounds, Random123's philox4x32_R<7>: the minimum Crush-resistant round count; csrc/philox.cuh says
 * why): for a logical row-major (rows, n) tensor
 *     w[0..3] = philox4x32_7(counter = (c >> 4, r, site, step), key = seed);   e = c & 15, i = e >> 2, j = e & 3
 *     keep(r, c)  <=>  (((byte j of w[i]) << 8 | (byte j of w[i ^ 1])) & 0x7fff)  >=  thr
 * with thr = round(p * 32768) <= 0x7c00 (p <= 0.96875) and kept values multiplied by scale = 32768 / (32768 - thr): one call
 * serves 16 columns, and 15-bit lanes let the kernels compare two of them with one half2 instruction (csrc/philox.cuh).  `state` is a device array
 * {uint64 seed, uint64 step}; lasr_rng_advance (one tiny kernel, CUDA-graph capturable) increments step, so every optimizer
 * step -- every replay of a captured step -- draws fresh masks.  Masks are never stored: lasr_gemm / lasr_layernorm_bwd_drop
 * evaluate them in their epilogues, the backward pass regenerates them from the same (step, site, row, column).
 *   lasr_dropout: y[r,c] = keep * scale * x[r,c] as a stand-alone pass (x fp32|bf16 -> y fp32|bf16; in place allowed when the
 *   dtypes agree) for the sites that sit behind no GEMM: pos_emb, the CTC head's input (fused with the operand cast), the
 *   decoder's embedded input and its gradient, attention probabilities when an attention dropout rate is non-zero.
 *   lasr_philox_raw: known-answer hook -- out[0..3] = philox4x32 with `rounds` (10 = the Random123 kat_vectors, 7 = the
 *   masks) rounds of counter ctr_key[0..3], key ctr_key[4..5] (device pointers).
 * ------------------------------------------------------------------------------------------------ */
int lasr_rng_advance(void* state, void* stream);
int lasr_philox_raw(const uint32_t* ctr_key, uint32_t* out, int rounds, void* stream);
int lasr_dropout(const void* x, int x_dtype, int64_t ldx, void* y, int y_dtype, int64_t ldy, int64_t rows, int cols,
                 const void* state, uint32_t site, uint32_t thr, float scale, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Casts / relayouts (weights fp32 master -> bf16 operand copies; conv weight permutations and the
 * inverse scatter of their gradients).  permute4d: dst[i.ds] (+)= src[i.ss] over a 4-D index space.
 * ------------------------------------------------------------------------------------------------ */
int lasr_cast_f32_bf16(const float* src, void* dst, int64_t n, void* stream);
int lasr_permute4d(const void* src, int src_dtype, void* dst, int dst_dtype, const int64_t* n, const int64_t* src_strides,
                   const int64_t* dst_strides, int accumulate, void* stream);

/* dh = scale * da * act'(saved) (saved = pre-activation for swish, activation output for relu), dbias += colsum(dh).
 * Backward of the fused bias+activation GEMM epilogue (nets/feed_forward.py:18-19, nn.Linear biases).
 * dh may be NULL for act = none (bias gradient only). */
int lasr_act_bwd(const void* da, int64_t ldda, const void* saved, int64_t lds, void* dh, int64_t lddh, float* dbias, int rows,
                 int cols, int act, float scale, int dtype, void* stream);

/* q + pos_bias_u, q + pos_bias_v (nets/attention.py:135-139) and the backward
 * (dq = dqu + dqv, du += colsum(dqu), dv += colsum(dqv), optional dqbias += colsum(dq): linear_q's bias gradient). */
int lasr_pos_bias_fwd(const void* q, int64_t ldq, const float* u, const float* v, void* qu, void* qv, int64_t ldo, int rows,
                      int d, int dtype, void* stream);
int lasr_pos_bias_bwd(const void* dqu, const void* dqv, int64_t ldi, void* dq, int64_t ldq, float* du, float* dv, float* dqbias,
                      int rows, int d, int dtype, void* stream);

/* Decoder input embedding: out[b,l] = emb[tokens[b,l]] * scale + pe[l] (nets/transformer_decoder.py:77-78,
 * nets/positional_encoding.py:49-56); backward scatter-adds scale*dout into demb (red.add). */
int lasr_embed_fwd(const int64_t* tokens, int L, const float* emb, const float* pe, float* out, int B, int d, float scale,
                   void* stream);
int lasr_embed_bwd(const int64_t* tokens, const float* dout, float* demb, int64_t rows, int d, float scale, void* stream);

/* x[i] *= *scalar (device scalar): applies autograd's upstream gradient to a loss-gradient buffer without a host sync. */
int lasr_scale_by_scalar(void* x, int dtype, int64_t n, const float* scalar, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Conformer convolution-module middle: GLU -> depthwise Conv1d(k=15,pad 7) -> BatchNorm1d -> Swish
 * (nets/conformer_convolution.py:49-53) on (B,T',C) channel-contiguous tensors, and its backward.
 *   y2 (B*T', 2d) = pointwise_conv1 output (value half | gate half), row stride ldy
 *   z  (B*T', d) fp32 = depthwise output;  partial: B*ceil(T'/32)*2*d floats of per-chunk sum / sum-sq
 *   bn_finalize: training=1 -> batch statistics over ALL B*T' frames (padding included, quirk Q2) +
 *                running-stat update (momentum, unbiased var, num_batches_tracked += 1);
 *                training=0 -> mean/rstd from the running statistics.
 *   bwd_stats : partial (ceil(rows/32)*2*d) -> sums[0:d] = sum du, sums[d:2d] = sum du*zhat; dgamma/dbeta +=
 *   dwconv_glu_bwd: dy2 (B*T',2d), dw (d,15) += , dbias (d) += , optional colsum (2d) += sum_rows dy2
 *                   (pointwise_conv1's bias gradient, taken while the rows are on chip); optional wpartial
 *                   (B*ceil(T'/32)*18*d floats): per-CTA partials + a second reduction kernel instead of atomics
 *                   (deterministic, and no same-address contention on the 16 KB of depthwise gradients)
 * ------------------------------------------------------------------------------------------------ */
int lasr_glu_dwconv_fwd(const void* y2, int dtype, int64_t ldy, const float* w, const float* bias, float* z, float* partial,
                        int B, int T, int d, void* stream);
/* glu_dwconv_fwd_lens: the same with per-utterance lengths lens (B,) int64 (sub-sampled frames, clamped to [0,T]): GLU outputs
 * of rows t >= lens[b] read as zero, the Conv1d zero padding of a batch-1 call on the utterance cut to lens[b] frames.  Rows
 * t < lens[b] of z then do not depend on the padded rows; rows t >= lens[b] hold finite values.  Inference only: no backward. */
int lasr_glu_dwconv_fwd_lens(const void* y2, int dtype, int64_t ldy, const float* w, const float* bias, float* z, float* partial,
                             int B, int T, int d, const int64_t* lens, void* stream);
int lasr_bn_finalize(const float* partial, int nblk, int d, int64_t count, float eps, float momentum, float* mean, float* rstd,
                     float* running_mean, float* running_var, int64_t* num_batches_tracked, int training, void* stream);
int lasr_bn_swish_fwd(const float* z, const float* mean, const float* rstd, const float* gamma, const float* beta, void* a,
                      int dtype, int64_t rows, int d, void* stream);
int lasr_bn_swish_bwd_stats(const void* da, int dtype, const float* z, const float* mean, const float* rstd, const float* gamma,
                            const float* beta, float* partial, float* sums, float* dgamma, float* dbeta, int64_t rows, int d,
                            void* stream);
int lasr_dwconv_glu_bwd(const void* da, const float* z, const void* y2, int dtype, int64_t ldy, const float* mean, const float* rstd,
                        const float* gamma, const float* beta, const float* sums, const float* w, void* dy2, int64_t lddy, float* dw,
                        float* dbias, float* colsum, float* wpartial, int B, int T, int d, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Conv2d subsampling (nets/subsampling.py:32-35,42-46), channel-last.
 *   conv1_fwd : x (B,T,F) fp32 -> h1 (B,T1,F1,d) = relu(conv3x3 s2), T1=(T-3)/2+1, F1=(F-3)/2+1
 *   conv1_bwd : dw (d,1,3,3) += , dbias += from dh1 (already ReLU-masked)
 *   im2col_s2 : h1 -> col (B*T2*F2, 9d), K index (kh,kw,c); conv2 itself is lasr_gemm on col
 *   col2im_s2_relu : dh1 = relu'(h1) * gather(dcol)
 * ------------------------------------------------------------------------------------------------ */
int lasr_conv1_fwd(const float* x, const float* w, const float* bias, void* h1, int dtype, int B, int T, int F, int d, void* stream);
int lasr_conv1_bwd(const float* x, const void* dh1, int dtype, float* dw, float* dbias, int B, int T, int F, int d, void* stream);
int lasr_im2col_s2(const void* h1, void* col, int dtype, int B, int T1, int F1, int d, void* stream);
int lasr_col2im_s2_relu(const void* dcol, const void* h1, void* dh1, int dtype, int B, int T1, int F1, int d, void* stream);

/* Parity-plane front end (bf16 / tcgen05 mode): conv1 writes h1p (B,4,U*V,d) with t1 = 2u+pt, f1 = 2v+pf, plane = pt*2+pf,
 * U = ceil(T1/2), V = ceil(F1/2), slots without a (t1,f1) zero; conv2 (nets/subsampling.py:33-34) then runs as an implicit
 * GEMM whose operand tiles are dense TMA boxes at a per-tap row offset -- no im2col / col2im buffers.
 *   conv2_fwd  : h2p (B, T2*V, d) bf16 = relu(conv3x3 s2 + bias); slot f2 = V-1 of every t2 row is padding (never read)
 *   conv2_dgrad: dh1p (B,4,U*V,d) = relu'(h1p) * conv2^T(dy2p); dy2p (B, T2*V, d) bf16 with the padding slot ZERO
 *   conv2_wgrad: dw2k (d, 9d) fp32 (co, kh, kw, ci) += dy2p^T * h1p patches
 *   conv1_bwd_planes: conv1 weight / bias gradient from dh1p */
int lasr_conv1_fwd_planes(const float* x, const float* w, const float* bias, void* h1p, int B, int T, int F, int d, void* stream);
int lasr_conv1_bwd_planes(const float* x, const void* dh1p, float* dw, float* dbias, int B, int T, int F, int d, void* stream);
int lasr_conv2_fwd(const void* h1p, const void* w2k, const float* bias, void* h2p, int B, int T, int F, int d, void* stream);
int lasr_conv2_dgrad(const void* dy2p, const void* w2k, const void* h1p, void* dh1p, int B, int T, int F, int d, void* stream);
int lasr_conv2_wgrad(const void* dy2p, const void* h1p, float* dw2k, int B, int T, int F, int d, void* stream);


/* ------------------------------------------------------------------------------------------------
 * Attention score post-processing (nets/attention.py:46-59,99-118,145-152): legacy rel_shift of bd
 * (NULL for plain attention) + scale + key/causal mask (-1e38 fill) + softmax, and the backward
 * (dscores = p*(dp - sum p*dp)*scale; dbd = inverse shift of dscores, NULL for plain attention).
 * ac/bd/dprobs (B,H,Tq,ld) of s_dtype: fp32, or bf16 when probs are bf16 (what torch autocast's matmul hands to the softmax;
 * halves the score traffic); probs/dscores/dbd fp32|bf16 (B,H,Tq,ld); columns [Tk,ld) are zeroed.
 * mask_mode: 0 none | 1 klen=lens[b] | 2 klen=lens[b]+1 | 3 klen=#{j: 4j<lens[b]} (encoder sub-sampled mask) |
 *            4 klen=lens[b] with the legacy shift run over klen instead of Tk (forward only, no backward counterpart):
 *              bdshift[i,j] = bd[i, klen-1-(i-j)] (j <= i) | 0 (j == i+1) | bd[i+1, j-i-2] (i+1 < j < klen), keys j >= klen -1e38;
 *              rows i < klen then equal the maskless batch-1 call on the utterance cut to klen frames (per-utterance inference
 *              on a padded batch), rows i >= klen get finite values without the rel-pos term.
 * Row width: ld even, Tk <= ld <= 16384 (T' = 16384 sub-sampled frames, about 10.9 minutes of audio at a 10 ms frame shift);
 * a larger ld returns LASR_ERR_BAD_ARG with a message naming the bound.  ld <= 1024 runs one warp per row, wider rows one
 * 512-thread CTA per row (B*H*Tq <= 2^31 - 1 rows); element offsets are 64-bit, so a tensor may exceed 2^31 elements.
 * A row's results do not depend on ld within either range.
 * ------------------------------------------------------------------------------------------------ */
int lasr_attn_softmax_fwd(const void* ac, const void* bd, int s_dtype, void* probs, int p_dtype, const int64_t* lens, int mask_mode,
                          int causal, float scale, int B, int H, int Tq, int Tk, int ld, void* stream);
int lasr_attn_softmax_bwd(const void* probs, const void* dprobs, int s_dtype, void* dscores, void* dbd, int dtype, float scale, int B,
                          int H, int Tq, int Tk, int ld, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused relative-position self-attention forward (nets/attention.py:99-154: matrix_ac, matrix_bd, the legacy rel_shift,
 * scale, key-padding masked_fill(-1e38), softmax, probs . V) in one tcgen05 kernel for bf16 operands:
 *   qu = q + pos_bias_u, qv = q + pos_bias_v : (B*T, H*dk) rows of stride ldq;  k, v : (B*T, H*dk) views, row stride ldkv;
 *   pos = linear_pos(pos_emb) : (T, H*dk), row stride ldp (broadcast over the batch)
 *   probs (B,H,T,ld) bf16 (saved for the backward pass; columns [T,ld) zeroed), o (B*T, H*dk) bf16, row stride ldo.
 * Replaces lasr_gemm x2 + lasr_attn_softmax_fwd + lasr_gemm for T <= 320, dk == 64 (lasr_rel_attn_fwd_supported);
 * other shapes return LASR_ERR_UNSUPPORTED and the caller keeps the unfused sequence.  mask_mode as lasr_attn_softmax_fwd.
 * ------------------------------------------------------------------------------------------------ */
int lasr_rel_attn_fwd_supported(int T, int dk);
void lasr_rel_attn_fwd_set_trace(void* buf); /* developer aid: 16 clock64 stamps per CTA (NULL = off) */
int lasr_rel_attn_fwd(const void* qu, const void* qv, long ldq, const void* k, const void* v, long ldkv, const void* pos, long ldp,
                      void* probs, int ld, void* o, long ldo, const int64_t* lens, int mask_mode, float scale, int B, int H, int T,
                      int dk, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Attention backward, the two contractions that consume one (B,H,Tq,Tk) gradient tensor X (autograd backward of
 * nets/attention.py:46-59 and :120-154 -- matrix_ac / matrix_bd), in ONE tcgen05 kernel that streams X through HBM once:
 *     dl[b, i, 64h:64h+64] = sum_j X[b,h,i,j] r[b, j, 64h:]          X = dscores: r = k,   dl = d(q + pos_bias_u)
 *     dr[b, j, 64h:64h+64] = sum_i X[b,h,i,j] l[b, i, 64h:]          X = dscores: l = q+u, dr = dk
 *   X (B,H,Tq,ldx) bf16 (columns [Tk,ldx) are never read); r: (B*Tk, *) rows of stride ldr, or ONE (Tk, *) matrix shared by
 *   every utterance when r_batched = 0 (X = dbd: r = linear_pos(pos_emb)); l, dl: (B*Tq, *) rows; dr: bf16 (B*Tk, *) rows, or --
 *   reduce_b = 1 -- fp32 (Tk, *) rows that RECEIVE (+=) the sum over the batch (X = dbd: l = q + pos_bias_v, dr = d pos).
 *   colsum (H*64 floats, may be NULL; reduce_b = 0 only) += column sums of dr over (b, j): the bias gradient of the projection
 *   that produced r.  Replaces two batched lasr_gemm launches for dk == 64, Tk <= 320 (lasr_attn_bwd_pair_supported).
 * ------------------------------------------------------------------------------------------------ */
int lasr_attn_bwd_pair_supported(int Tk, int dk);
int lasr_attn_bwd_pair(const void* x, int64_t ldx, const void* r, int64_t ldr, int r_batched, const void* l, int64_t ldl, void* dl, int64_t lddl,
                       void* dr, int64_t lddr, int reduce_b, float* colsum, int B, int H, int Tq, int Tk, int dk, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Label-smoothed KL on the decoder logits, forward + gradient (criterions/hybrid_ctc_attn.py:49-64;
 * targets built on the fly from ys/ylens as models/u2.py:323-328), and the hybrid mix (:78).
 * row_loss: B*(lmax+1) floats.  hybrid_combine: out[0]=loss, out[1]=ctc term, out[2]=attention term.
 * ------------------------------------------------------------------------------------------------ */
int lasr_lsmooth_kl_fwdbwd(const void* logits, int dtype, int64_t ldl, const int64_t* ys, const int64_t* ylens, int B, int lmax, int V,
                           float smoothing, float grad_scale, const float* upstream, float* row_loss, void* grad, int64_t ldg,
                           void* stream);
int lasr_hybrid_combine(const float* nll, int B, const float* row_kl, int M, float ctc_weight, float* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused optimizer tail over flat buffers (trainer.py:153-171, optims/noam.py:33-46, optims/adam.py:27-34):
 * global-norm clip + NaN-skip + Noam LR + Adam, no host sync.  state: 8 floats {step, grad_norm, lr,
 * skipped, grad_scale,...}; workspace: 1024 floats.
 * ------------------------------------------------------------------------------------------------ */
int lasr_clip_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float grad_mult,
                        float max_norm, float beta1, float beta2, float eps, float weight_decay, float noam_factor, float model_dim,
                        float warmup, float fixed_lr, float* state, float* workspace, void* stream);
int lasr_zero(void* ptr, size_t bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Inference (models/u2.py:221-317, nets/ctc.py:25-26).
 *   logsoftmax_topk : per row lse (optional), full log-softmax (optional, fp32, row stride ldf) and the K best classes in
 *                     (log-prob descending, index ascending) order: top_val (rows,K) fp32 log-probs, top_idx (rows,K) int32.
 *                     K = 1 is greedy CTC's argmax; K = beam is the per-frame prune of the prefix search (u2.py:230).
 *   gather_logp     : out[r] = logits[r, tokens[r]] - lse[r]  (attention-rescoring lookups, u2.py:306-310).
 *   ctc_prefix_beam_search : HOST function (no device work): u2.py:224-261 on host copies of top_val / top_idx for ONE
 *                     utterance; float64 arithmetic in the reference's operation order, insertion-ordered prefix map, stable
 *                     sort.  Outputs up to `beam` hypotheses best first: tokens (beam,max_len) padded -1, lengths, scores.
 *   ctc_prefix_beam_search_batch : the same search on the DEVICE for a ragged batch in one launch, no host synchronisation,
 *                     deterministic.  top_val / top_idx (B*Tmax, K) as logsoftmax_topk emits them (utterance b at rows
 *                     [b*Tmax, b*Tmax + frames[b])), frames (B,) int64 (clamped to [0,Tmax]).  Outputs: tokens
 *                     (B,beam,max_len) padded -1 (max_len >= Tmax), lengths (B,beam), float64 scores (B,beam) (-inf beyond
 *                     the count), hypothesis counts (B,).  1 <= K <= 64, 1 <= beam <= 32.  workspace: at least
 *                     ctc_prefix_beam_search_batch_workspace(B, Tmax, beam) bytes (the prefix-node pools).  Float64 with CUDA's
 *                     exp / log (<= 1 ulp): scores may differ from the host function's in the last bits, and two hypotheses
 *                     whose scores lie within a few ulps may come out in the other order.
 * CTC Viterbi forced alignment (token timestamps) of a ragged batch: declared in include/lasr_align.h.
 * Kaldi-compatible log-mel filterbank features of a padded batch of waveforms: declared in include/lasr_fbank.h.
 * ------------------------------------------------------------------------------------------------ */
int lasr_logsoftmax_topk(const void* logits, int dtype, int64_t ld, int64_t rows, int V, int K, float* lse, float* logp_full,
                         int64_t ldf, float* top_val, int32_t* top_idx, void* stream);
int lasr_gather_logp(const void* logits, int dtype, int64_t ld, const float* lse, const int64_t* tokens, float* out, int64_t rows, int V,
                     void* stream);
int lasr_ctc_prefix_beam_search(const float* topk_logp, const int32_t* topk_idx, int frames, int K, int beam, int blank,
                                int32_t* out_tokens, int32_t* out_lens, double* out_scores, int max_len, int32_t* n_out);
size_t lasr_ctc_prefix_beam_search_batch_workspace(int B, int Tmax, int beam);
int lasr_ctc_prefix_beam_search_batch(const float* top_val, const int32_t* top_idx, const int64_t* frames, int B, int Tmax, int K, int beam,
                                      int blank, int32_t* out_tokens, int32_t* out_lens, double* out_scores, int32_t* out_n, int max_len,
                                      void* workspace, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * SpecAugment on a padded batch (utils/transform/spec_augment.py:19-125; SURVEY 8f N3), out of place.
 *   x, y   : (B, ld_batch / F rows, F) fp32, utterance b occupies rows [0, T_b)
 *   params : int32 (B, lasr_spec_augment_npar()) = {T_b, center, warped, n_freq, n_time, 8 x (lo, hi) frequency masks,
 *            8 x (lo, hi) time masks}; center < 0 = no time warp.  The decisions are drawn on the host in the reference's
 *            RNG order; the kernel reproduces PIL's BICUBIC resize (mode "F") bit for bit and fills the masks, in order, with
 *            the mean of the array at that moment (replace_with_zero = 0) or zero.
 * ------------------------------------------------------------------------------------------------ */
int lasr_spec_augment_npar(void);
int lasr_spec_augment(const float* x, float* y, int64_t ld_batch, int F, const int32_t* params, int B, int replace_with_zero,
                      void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LASR_H */
