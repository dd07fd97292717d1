// Attention score post-processing, fused: legacy rel_shift + scale + key-padding / causal mask + softmax
// (nets/attention.py:46-59,99-118,145-152) and the matching backward.
//
// The dense contractions (Q.K^T, Q.P^T, probs.V and their transposes) run on the tcgen05 GEMM; these kernels
// do everything between them in ONE pass per direction, one warp per score row held in registers:
//   fwd : s[i,j] = (ac[i,j] + bdshift[i,j]) * scale ; masked -> -1e38 ; p = softmax_j(s)   (bf16/fp32 out)
//         bdshift[i,j] = bd[i, Tk-1-(i-j)] (j <= i) | 0 (j == i+1) | bd[i+1, j-i-2] (j > i+1)      (quirk Q1)
//   bwd : ds = p * (dp - sum_j p*dp) * scale  -> dac ; dbd = the same values scattered through the inverse shift (same pass)
// Key mask: key j of batch b is valid iff j < klen(b);  klen mode: 0 none, 1 lens[b], 2 lens[b]+1,
// 3 #{j : 4j < lens[b]} (the encoder's mask[:, :-2:2][:, :-2:2] of a padding mask, nets/transformer_encoder.py:118),
// 4 lens[b] with the legacy shift taken over klen instead of Tk (per-utterance inference on a padded batch: every valid row equals
// the maskless batch-1 call on the utterance cut to its length; rows i >= klen get finite values without the rel-pos term).
// Masked scores are -1e38 exactly like masked_fill (no -inf, no post-softmax zeroing: quirk Q4).
#include "common.cuh"

namespace lasr {

constexpr int SM_MAXP = 16;  // column pairs per lane -> Tk <= 1024
constexpr float MASK_FILL = -1e38f;

__device__ __forceinline__ int key_len(const int64_t* lens, int mode, int b, int Tk) {
    if (mode == 0 || !lens) return Tk;
    const long l = lens[b];
    long k = l;
    if (mode == 2) k = l + 1;
    else if (mode == 3) k = (l + 3) / 4;
    return (int)(k < Tk ? (k < 0 ? 0 : k) : Tk);
}

template <typename TP> __device__ __forceinline__ void store_pair(TP* p, float a, float b);
template <> __device__ __forceinline__ void store_pair<float>(float* p, float a, float b) { *reinterpret_cast<float2*>(p) = make_float2(a, b); }
template <> __device__ __forceinline__ void store_pair<bf16>(bf16* p, float a, float b) {
    *reinterpret_cast<__nv_bfloat162*>(p) = __floats2bfloat162_rn(a, b);
}
template <typename TP> __device__ __forceinline__ float2 load_pair(const TP* p);
template <> __device__ __forceinline__ float2 load_pair<float>(const float* p) { return *reinterpret_cast<const float2*>(p); }
template <> __device__ __forceinline__ float2 load_pair<bf16>(const bf16* p) {
    const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(p);
    return make_float2(__low2float(h), __high2float(h));
}

// One warp per score row; lane l owns the column pairs (2l + 64e, 2l + 64e + 1), e < NP (ld <= 64 NP): 64-bit loads of ac,
// 32/64-bit stores of the probabilities, NP sized to the problem so the kernel runs at full occupancy.  ld must be even.
template <typename TP, typename TS, int NP, bool RAGGED = false>
__global__ void __launch_bounds__(256) attn_softmax_fwd_kernel(const TS* __restrict__ ac, const TS* __restrict__ bd,
                                                               TP* __restrict__ probs, const int64_t* __restrict__ lens,
                                                               int mask_mode, int causal, float scale, int B, int H, int Tq,
                                                               int Tk, int ld) {
    LASR_PDL_SYNC();
    const int lane = threadIdx.x & 31;
    const long row = (long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= (long)B * H * Tq) return;
    const int i = (int)(row % Tq);
    const int b = (int)(row / ((long)H * Tq));
    const int klen = RAGGED ? key_len(lens, 1, b, Tk) : key_len(lens, mask_mode, b, Tk);
    const TS* ar = ac + row * ld;
    const TS* br = bd ? bd + row * ld : nullptr;  // bd row i of the same (b,h); row i+1 is br + ld
    float2 s[NP];
    float mx = -INFINITY;
#pragma unroll
    for (int e = 0; e < NP; ++e) {
        const int j = 2 * lane + 64 * e;
        s[e] = make_float2(-INFINITY, -INFINITY);
        if (j < Tk) {
            float2 v = load_pair<TS>(ar + j);
            const bool two = j + 1 < Tk;
            if (RAGGED) {
                // the shift over klen: bd[i, klen-1-(i-j)] (j <= i) | 0 (j == i+1) | bd[i+1, j-i-2] (i+1 < j < klen)
                if (br && i < klen) {
                    if (j < klen) v.x += (j <= i) ? to_f32<TS>(br[klen - 1 - i + j]) : ((j > i + 1) ? to_f32<TS>(br[ld + j - i - 2]) : 0.f);
                    if (j + 1 < klen) v.y += (j + 1 <= i) ? to_f32<TS>(br[klen - i + j]) : ((j > i) ? to_f32<TS>(br[ld + j - i - 1]) : 0.f);
                }
            } else if (br) {
                // legacy rel_shift: bd[i, Tk-1-(i-j)] (j <= i) | 0 (j == i+1) | bd[i+1, j-i-2] (j > i+1)
                v.x += (j <= i) ? to_f32<TS>(br[Tk - 1 - i + j]) : ((j > i + 1) ? to_f32<TS>(br[ld + j - i - 2]) : 0.f);
                if (two) v.y += (j + 1 <= i) ? to_f32<TS>(br[Tk - i + j]) : ((j > i) ? to_f32<TS>(br[ld + j - i - 1]) : 0.f);
            }
            v.x *= scale; v.y *= scale;
            if (j >= klen || (causal && j > i)) v.x = MASK_FILL;
            if (j + 1 >= klen || (causal && j + 1 > i)) v.y = MASK_FILL;
            if (!two) v.y = -INFINITY;
            s[e] = v;
            mx = fmaxf(mx, fmaxf(v.x, v.y));
        }
    }
    mx = warp_max(mx);
    float sum = 0.f;
#pragma unroll
    for (int e = 0; e < NP; ++e) {
        s[e].x = expf(s[e].x - mx);  // exp(-inf) = 0 for columns beyond Tk
        s[e].y = expf(s[e].y - mx);
        sum += s[e].x + s[e].y;
    }
    sum = warp_sum(sum);
    const float inv = 1.f / sum;
    TP* pr = probs + row * ld;
#pragma unroll
    for (int e = 0; e < NP; ++e) {
        const int j = 2 * lane + 64 * e;
        if (j < ld) store_pair<TP>(pr + j, s[e].x * inv, s[e].y * inv);  // columns [Tk, ld) get exact zeros
    }
}

// ds = p * (dp - sum_j p dp) * scale, written to dsc in place of the score gradient AND (rel-pos attention) scattered through
// the inverse of the legacy shift into dbd: ds[i, j <= i] -> dbd[i, Tk-1-i+j], ds[i, j >= i+2] -> dbd[i+1, j-i-2]; every
// element of a dbd row is written exactly once (row r = [tail of ds row r-1 | head of ds row r]; row 0 starts with zeros).
template <typename TP, typename TS, int NP>
__global__ void __launch_bounds__(256) attn_softmax_bwd_kernel(const TP* __restrict__ probs, const TS* __restrict__ dprobs,
                                                               TP* __restrict__ dsc, TP* __restrict__ dbd, float scale, long rows,
                                                               int Tq, int Tk, int ld) {
    LASR_PDL_SYNC();
    const int lane = threadIdx.x & 31;
    const long row = (long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= rows) return;
    const TP* pr = probs + row * ld;
    const TS* dr = dprobs + row * ld;
    float2 p[NP], g[NP];
    float dot = 0.f;
#pragma unroll
    for (int e = 0; e < NP; ++e) {
        const int j = 2 * lane + 64 * e;
        p[e] = make_float2(0.f, 0.f); g[e] = make_float2(0.f, 0.f);
        if (j < Tk) {
            p[e] = load_pair<TP>(pr + j);
            g[e] = load_pair<TS>(dr + j);
            if (j + 1 >= Tk) { p[e].y = 0.f; g[e].y = 0.f; }
            dot += p[e].x * g[e].x + p[e].y * g[e].y;
        }
    }
    dot = warp_sum(dot);
    TP* o = dsc + row * ld;
    const int i = (int)(row % Tq);
    TP* d0 = dbd ? dbd + row * ld : nullptr;  // dbd row i; row i+1 = d0 + ld
#pragma unroll
    for (int e = 0; e < NP; ++e) {
        const int j = 2 * lane + 64 * e;
        if (j < ld) {
            const float x = p[e].x * (g[e].x - dot) * scale, y = p[e].y * (g[e].y - dot) * scale;  // zero beyond Tk
            store_pair<TP>(o + j, x, y);
            if (d0) {
                if (j < Tk) {
                    if (j <= i) d0[Tk - 1 - i + j] = from_f32<TP>(x);
                    else if (j > i + 1) d0[ld + j - i - 2] = from_f32<TP>(x);
                } else {
                    d0[j] = from_f32<TP>(0.f);  // padding columns of dbd row i
                }
                if (j + 1 < Tk) {
                    if (j + 1 <= i) d0[Tk - i + j] = from_f32<TP>(y);
                    else if (j > i) d0[ld + j - i - 1] = from_f32<TP>(y);
                } else if (j + 1 < ld) {
                    d0[j + 1] = from_f32<TP>(0.f);
                }
                if (i == 0 && j < Tk - 1) {  // dbd row 0, columns [0, Tk-2]: no source row
                    d0[j] = from_f32<TP>(0.f);
                    if (j + 1 < Tk - 1) d0[j + 1] = from_f32<TP>(0.f);
                }
            }
        }
    }
}

}  // namespace lasr

extern "C" {
using namespace lasr;

// NP is chosen from the row width ld, not from Tk: a lane writes only columns j < 64 NP, and every column of [Tk, ld) must be
// zeroed.  The bucket edges are multiples of 64, so ld = ceil(Tk, 8) or ceil(Tk, 64) selects the same NP as Tk would.
#define LASR_SM_DISPATCH(KERNEL, TP, TS, ...)                                        \
    do {                                                                             \
        if (ld <= 64) launch_pdl(KERNEL<TP, TS, 1>, grid, 256, 0, st, __VA_ARGS__);          \
        else if (ld <= 128) launch_pdl(KERNEL<TP, TS, 2>, grid, 256, 0, st, __VA_ARGS__);    \
        else if (ld <= 320) launch_pdl(KERNEL<TP, TS, 5>, grid, 256, 0, st, __VA_ARGS__);    \
        else if (ld <= 448) launch_pdl(KERNEL<TP, TS, 7>, grid, 256, 0, st, __VA_ARGS__);    \
        else launch_pdl(KERNEL<TP, TS, SM_MAXP>, grid, 256, 0, st, __VA_ARGS__);             \
    } while (0)

// mask mode 4: the RAGGED instantiations of the forward kernel
#define LASR_SM_DISPATCH_RAGGED(TP, TS, ...)                                                               \
    do {                                                                                                    \
        if (ld <= 64) launch_pdl(attn_softmax_fwd_kernel<TP, TS, 1, true>, grid, 256, 0, st, __VA_ARGS__);          \
        else if (ld <= 128) launch_pdl(attn_softmax_fwd_kernel<TP, TS, 2, true>, grid, 256, 0, st, __VA_ARGS__);    \
        else if (ld <= 320) launch_pdl(attn_softmax_fwd_kernel<TP, TS, 5, true>, grid, 256, 0, st, __VA_ARGS__);    \
        else if (ld <= 448) launch_pdl(attn_softmax_fwd_kernel<TP, TS, 7, true>, grid, 256, 0, st, __VA_ARGS__);    \
        else launch_pdl(attn_softmax_fwd_kernel<TP, TS, SM_MAXP, true>, grid, 256, 0, st, __VA_ARGS__);             \
    } while (0)

int lasr_attn_softmax_fwd(const void* ac, const void* bd, int s_dtype, void* probs, int p_dtype, const int64_t* lens, int mask_mode,
                          int causal, float scale, int B, int H, int Tq, int Tk, int ld, void* stream) {
    LASR_REQUIRE(ac && probs && B > 0 && H > 0 && Tq > 0 && Tk > 0 && ld >= Tk && ld <= 64 * SM_MAXP && ld % 2 == 0,
                 "attn_softmax_fwd: bad args (Tk <= ld <= 1024, ld even)");
    LASR_REQUIRE(!bd || Tq == Tk, "attn_softmax_fwd: rel_shift needs Tq == Tk");
    LASR_REQUIRE(mask_mode >= 0 && mask_mode <= 4 && (mask_mode == 0 || lens), "attn_softmax_fwd: bad mask mode");
    LASR_REQUIRE(((uintptr_t)ac & 7) == 0 && ((uintptr_t)probs & 7) == 0, "attn_softmax_fwd: unaligned");
    const long rows = (long)B * H * Tq;
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = ceil_div(rows, 8);
    if (mask_mode == 4) {
        if (p_dtype == LASR_F32 && s_dtype == LASR_F32)
            LASR_SM_DISPATCH_RAGGED(float, float, (const float*)ac, (const float*)bd, (float*)probs, lens, mask_mode, causal, scale, B, H, Tq, Tk, ld);
        else if (p_dtype == LASR_BF16 && s_dtype == LASR_F32)
            LASR_SM_DISPATCH_RAGGED(bf16, float, (const float*)ac, (const float*)bd, (bf16*)probs, lens, mask_mode, causal, scale, B, H, Tq, Tk, ld);
        else if (p_dtype == LASR_BF16 && s_dtype == LASR_BF16)
            LASR_SM_DISPATCH_RAGGED(bf16, bf16, (const bf16*)ac, (const bf16*)bd, (bf16*)probs, lens, mask_mode, causal, scale, B, H, Tq, Tk, ld);
        else { set_error("attn_softmax_fwd: unsupported dtype combination"); return LASR_ERR_UNSUPPORTED; }
        return check_launch("attn_softmax_fwd");
    }
    if (p_dtype == LASR_F32 && s_dtype == LASR_F32)
        LASR_SM_DISPATCH(attn_softmax_fwd_kernel, float, float, (const float*)ac, (const float*)bd, (float*)probs, lens, mask_mode, causal, scale, B, H, Tq, Tk, ld);
    else if (p_dtype == LASR_BF16 && s_dtype == LASR_F32)
        LASR_SM_DISPATCH(attn_softmax_fwd_kernel, bf16, float, (const float*)ac, (const float*)bd, (bf16*)probs, lens, mask_mode, causal, scale, B, H, Tq, Tk, ld);
    else if (p_dtype == LASR_BF16 && s_dtype == LASR_BF16)
        LASR_SM_DISPATCH(attn_softmax_fwd_kernel, bf16, bf16, (const bf16*)ac, (const bf16*)bd, (bf16*)probs, lens, mask_mode, causal, scale, B, H, Tq, Tk, ld);
    else { set_error("attn_softmax_fwd: unsupported dtype combination"); return LASR_ERR_UNSUPPORTED; }
    return check_launch("attn_softmax_fwd");
}

int lasr_attn_softmax_bwd(const void* probs, const void* dprobs, int s_dtype, void* dscores, void* dbd, int dtype, float scale, int B,
                          int H, int Tq, int Tk, int ld, void* stream) {
    LASR_REQUIRE(probs && dprobs && dscores && B > 0 && H > 0 && Tq > 0 && Tk > 0 && ld >= Tk && ld <= 64 * SM_MAXP && ld % 2 == 0,
                 "attn_softmax_bwd: bad args");
    LASR_REQUIRE(!dbd || Tq == Tk, "attn_softmax_bwd: rel_shift needs Tq == Tk");
    LASR_REQUIRE(((uintptr_t)probs & 7) == 0 && ((uintptr_t)dprobs & 7) == 0 && ((uintptr_t)dscores & 7) == 0, "attn_softmax_bwd: unaligned");
    const long rows = (long)B * H * Tq;
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = ceil_div(rows, 8);
    if (dtype == LASR_F32 && s_dtype == LASR_F32)
        LASR_SM_DISPATCH(attn_softmax_bwd_kernel, float, float, (const float*)probs, (const float*)dprobs, (float*)dscores, (float*)dbd, scale, rows, Tq, Tk, ld);
    else if (dtype == LASR_BF16 && s_dtype == LASR_F32)
        LASR_SM_DISPATCH(attn_softmax_bwd_kernel, bf16, float, (const bf16*)probs, (const float*)dprobs, (bf16*)dscores, (bf16*)dbd, scale, rows, Tq, Tk, ld);
    else if (dtype == LASR_BF16 && s_dtype == LASR_BF16)
        LASR_SM_DISPATCH(attn_softmax_bwd_kernel, bf16, bf16, (const bf16*)probs, (const bf16*)dprobs, (bf16*)dscores, (bf16*)dbd, scale, rows, Tq, Tk, ld);
    else { set_error("attn_softmax_bwd: unsupported dtype combination"); return LASR_ERR_UNSUPPORTED; }
    return check_launch("attn_softmax_bwd");
}

}  // extern "C"
