// CTC Viterbi forced alignment of a ragged batch (lasr_ctc_forced_align, include/lasr_align.h): the single most likely CTC
// path of a known label sequence over the CTC head's log-probabilities (nets/ctc.py:25-26, log_softmax(ctc_lo(x))).  The
// reference ships no aligner; the definition below is this project's.
//
// One CTA per utterance.  S = 2L+1 extended states (z[2k] = blank, z[2k+1] = y[k]); thread `tid` owns the run of R states
// [tid*R, tid*R + R), R a power of two <= 32, so one 64-bit word holds its 2-bit back-pointers of a frame.  The lattice row
// delta lives in shared memory, transposed (state tid*R + j at word j*NT + tid: conflict-free), and is updated in place:
//   - each thread reads its left neighbour's top two states of the previous frame from a double-buffered boundary array,
//   - updates its own states in DESCENDING order (state s reads s-1 and s-2 before they are overwritten),
//   - publishes its new top two states, then one barrier per frame.
// The emissions of frame t+1 (R/2 label logits, the blank logit and lse) are loaded while frame t is computed.
// Arithmetic: e = float(logit) - lse (one fp32 subtraction), delta = max(predecessors) + e (one fp32 add); max is exact, so a
// float32 restatement reproduces every output bit for bit.
// Traceback: thread 0 walks the back-pointers from the end state; the per-frame log-probs are then filled by the whole CTA.
#include <cmath>

#include "common.cuh"
#include "../../include/lasr_align.h"

namespace lasr {

constexpr int AL_MAX_LABELS = 16383, AL_MAX_FRAMES = 16384;

struct AlCfg {
    int nt, r;  // threads per CTA, states per thread
};

// NT = clamp(roundup32(ceil(S / 8)), 32, 1024) threads, R = the power of two >= ceil(S / NT) (2 <= R <= 32): a warp of
// 4 states per thread at short transcripts, 8 states per thread up to S = 8192, 16 or 32 past it
static AlCfg al_config(int lmax) {
    const int S = 2 * lmax + 1;
    int nt = (S + 7) / 8;
    nt = (nt + 31) / 32 * 32;
    nt = nt < 32 ? 32 : (nt > 1024 ? 1024 : nt);
    int r = 2;
    while (r * nt < S) r *= 2;
    return AlCfg{nt, r};
}

static size_t al_smem_bytes(AlCfg c) {
    return (size_t)c.r * c.nt * sizeof(float) + (size_t)(c.r / 2) * c.nt * sizeof(int) + 2 * (size_t)c.nt * sizeof(float2);
}

template <typename T, int R>
__global__ void __launch_bounds__(1024) ctc_forced_align_kernel(const T* __restrict__ logits, long ld, const float* __restrict__ lse,
                                                                const int64_t* __restrict__ targets, const int64_t* __restrict__ tgt_len,
                                                                const int64_t* __restrict__ frames, int Tmax, int lmax, int V, int blank,
                                                                int32_t* __restrict__ out_state, float* __restrict__ out_logp,
                                                                float* __restrict__ out_score, int32_t* __restrict__ out_spans,
                                                                unsigned long long* __restrict__ bp_all) {
    constexpr int H = R / 2;  // label (odd) states per thread
    extern __shared__ __align__(16) uint8_t al_raw[];
    const int NT = blockDim.x, tid = threadIdx.x, b = blockIdx.x;
    float* sd = reinterpret_cast<float*>(al_raw);                      // [R][NT]   delta
    int* slab = reinterpret_cast<int*>(sd + (size_t)R * NT);           // [H][NT]   label of state tid*R + 2i + 1 (-1: none)
    float2* bnd = reinterpret_cast<float2*>(slab + (size_t)H * NT);    // [2][NT]   (delta[top], delta[top - 1]) per thread
    __shared__ int s_feasible;

    long Tb = frames[b];
    Tb = Tb < 0 ? 0 : (Tb > Tmax ? Tmax : Tb);
    long Lb = tgt_len[b];
    Lb = Lb < 0 ? 0 : (Lb > lmax ? lmax : Lb);
    const int S = 2 * (int)Lb + 1;
    const int s0 = tid * R;
    const int64_t* y = targets + (long)b * lmax;
    const T* lg = logits + (long)b * Tmax * ld;
    const float* ls = lse + (long)b * Tmax;
    unsigned long long* bp = bp_all + (long)b * Tmax * NT;

    // labels and the s-2 skip mask: state s0 + 2i + 1 (label k = s0/2 + i) may come from s - 2 when k >= 1 and y[k] != y[k-1]
    unsigned skip = 0;
#pragma unroll
    for (int i = 0; i < H; ++i) {
        const int k = s0 / 2 + i;
        int lab = -1;
        if (k < Lb) {
            const long v = y[k];
            lab = (v >= 0 && v < V) ? (int)v : -1;  // a label outside [0, V) has emission -inf
            if (k >= 1 && y[k - 1] != v) skip |= 1u << i;
        }
        slab[i * NT + tid] = lab;
    }
    const bool blank_ok = blank >= 0 && blank < V;

    // raw emissions of the current frame: H label logits, the blank logit, lse.  The label logit of frame t+1 is loaded into
    // the register of frame t's right after its last use, so one set of H registers carries the prefetch
    float el[H], eb = -INFINITY, lse_t = 0.f;
    auto lab_logit = [&](long t, int i) {
        const int lab = slab[i * NT + tid];
        return lab >= 0 ? to_f32<T>(lg[t * ld + lab]) : -INFINITY;
    };
    if (Tb > 0) {
#pragma unroll
        for (int i = 0; i < H; ++i) el[i] = lab_logit(0, i);
        eb = blank_ok ? to_f32<T>(lg[blank]) : -INFINITY;
        lse_t = ls[0];
    }

    for (long t = 0; t < Tb; ++t) {
        const bool more = t + 1 < Tb;
        const float cb = eb, clse = lse_t;
        if (more) {
            eb = blank_ok ? to_f32<T>(lg[(t + 1) * ld + blank]) : -INFINITY;
            lse_t = ls[t + 1];
        }
        const int par = (int)(t & 1);
        unsigned long long bits = 0ull;
        float top0, top1;  // new delta of states s0 + R - 1, s0 + R - 2
        if (t == 0) {
#pragma unroll
            for (int j = R - 1; j >= 0; --j) {
                const int s = s0 + j;
                const float e = (j & 1) ? el[j >> 1] - clse : cb - clse;
                if ((j & 1) && more) el[j >> 1] = lab_logit(t + 1, j >> 1);
                const float d = (s < 2 && s < S) ? e : -INFINITY;
                sd[j * NT + tid] = d;
                if (j == R - 1) top0 = d;
                if (j == R - 2) top1 = d;
            }
        } else {
            const float2 left = tid > 0 ? bnd[(par ^ 1) * NT + tid - 1] : make_float2(-INFINITY, -INFINITY);
            // sliding window over the old row, descending: a = old[j], c1 = old[j-1]
            float a = sd[(R - 1) * NT + tid];
            float c1 = sd[(R - 2) * NT + tid];
#pragma unroll
            for (int j = R - 1; j >= 0; --j) {
                const float c2 = j >= 2 ? sd[(j - 2) * NT + tid] : (j == 1 ? left.x : left.y);
                const int s = s0 + j;
                float best = a;
                unsigned p = 0;
                if (s >= 1 && c1 > best) { best = c1; p = 1; }
                if ((j & 1) && ((skip >> (j >> 1)) & 1u) && c2 > best) { best = c2; p = 2; }
                const float e = s < S ? ((j & 1) ? el[j >> 1] - clse : cb - clse) : -INFINITY;
                if ((j & 1) && more) el[j >> 1] = lab_logit(t + 1, j >> 1);
                const float d = best + e;
                sd[j * NT + tid] = d;
                bits |= (unsigned long long)p << (2 * j);
                if (j == R - 1) top0 = d;
                if (j == R - 2) top1 = d;
                a = c1;
                c1 = c2;
            }
            bp[t * NT + tid] = bits;
        }
        bnd[par * NT + tid] = make_float2(top0, top1);
        __syncthreads();
    }

    // ---- end state: the better of S-1 and S-2, a tie to S-1 (trailing blank)
    int32_t* st_row = out_state + (long)b * Tmax;
    float* lp_row = out_logp + (long)b * Tmax;
    int32_t* sp = out_spans + (long)b * lmax * 2;
    int end = S - 1;
    if (tid == 0) {
        float best = -INFINITY;
        if (Tb > 0) {
            best = sd[((S - 1) % R) * NT + (S - 1) / R];
            if (S >= 2) {
                const float d2 = sd[((S - 2) % R) * NT + (S - 2) / R];
                if (d2 > best) { best = d2; end = S - 2; }
            }
        }
        const bool ok = best > -INFINITY;
        s_feasible = ok;
        out_score[b] = ok ? best : -INFINITY;
    }
    __syncthreads();
    const bool ok = s_feasible != 0;
    for (long t = ok ? Tb + tid : tid; t < Tmax; t += NT) { st_row[t] = -1; lp_row[t] = -INFINITY; }
    for (long k = ok ? Lb + tid : tid; k < lmax; k += NT) { sp[2 * k] = -1; sp[2 * k + 1] = -1; }
    if (ok && tid == 0) {
        int s = end, cur_k = -1;
        for (long t = Tb - 1; t >= 0; --t) {
            st_row[t] = s;
            if (s & 1) {
                const int k = s >> 1;
                if (k != cur_k) { sp[2 * k + 1] = (int32_t)t; cur_k = k; }
                sp[2 * k] = (int32_t)t;
            }
            if (t > 0) {
                const unsigned long long w = bp[t * NT + s / R];
                s -= (int)((w >> (2 * (s % R))) & 3ull);
            }
        }
    }
    __syncthreads();
    if (ok) {
        for (long t = tid; t < Tb; t += NT) {
            const int s = st_row[t];
            const float x = (s & 1) ? to_f32<T>(lg[t * ld + (int)y[s >> 1]]) : to_f32<T>(lg[t * ld + blank]);
            lp_row[t] = x - ls[t];
        }
    }
}

template <typename T>
static void launch_align(AlCfg c, size_t smem, cudaStream_t st, int B, const void* logits, long ld, const float* lse,
                         const int64_t* targets, const int64_t* tgt_len, const int64_t* frames, int Tmax, int lmax, int V, int blank,
                         int32_t* state, float* logp, float* score, int32_t* spans, unsigned long long* bp) {
    void (*k)(const T*, long, const float*, const int64_t*, const int64_t*, const int64_t*, int, int, int, int, int32_t*, float*, float*,
              int32_t*, unsigned long long*);
    switch (c.r) {
        case 2: k = ctc_forced_align_kernel<T, 2>; break;
        case 4: k = ctc_forced_align_kernel<T, 4>; break;
        case 8: k = ctc_forced_align_kernel<T, 8>; break;
        case 16: k = ctc_forced_align_kernel<T, 16>; break;
        default: k = ctc_forced_align_kernel<T, 32>; break;
    }
    if (smem > 48 * 1024 && cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return;
    k<<<B, c.nt, smem, st>>>((const T*)logits, ld, lse, targets, tgt_len, frames, Tmax, lmax, V, blank, state, logp, score, spans, bp);
}

}  // namespace lasr

extern "C" {
using namespace lasr;

size_t lasr_ctc_forced_align_workspace(int B, int Tmax, int lmax) {
    if (B <= 0 || Tmax <= 0 || lmax < 0 || Tmax > AL_MAX_FRAMES || lmax > AL_MAX_LABELS) return 0;
    return (size_t)B * Tmax * al_config(lmax).nt * sizeof(unsigned long long);
}

int lasr_ctc_forced_align(const void* logits, int dtype, int64_t ld, const float* lse, const int64_t* targets, const int64_t* tgt_len,
                          const int64_t* frames, int B, int Tmax, int lmax, int V, int blank, int32_t* state, float* frame_logp,
                          float* score, int32_t* spans, void* workspace, size_t ws_bytes, void* stream) {
    LASR_REQUIRE(logits && lse && tgt_len && frames && state && frame_logp && score && B > 0 && Tmax > 0 && lmax >= 0 && V > 0 && ld >= V,
                 "ctc_forced_align: bad args");
    LASR_REQUIRE(lmax == 0 || (targets && spans), "ctc_forced_align: targets and spans are required when lmax > 0");
    LASR_REQUIRE(Tmax <= AL_MAX_FRAMES, "ctc_forced_align: Tmax %d exceeds the limit of %d frames", Tmax, AL_MAX_FRAMES);
    LASR_REQUIRE(lmax <= AL_MAX_LABELS, "ctc_forced_align: lmax %d exceeds the limit of %d labels", lmax, AL_MAX_LABELS);
    LASR_REQUIRE(blank >= 0 && blank < V, "ctc_forced_align: blank %d outside [0, V = %d)", blank, V);
    LASR_REQUIRE(workspace && ws_bytes >= lasr_ctc_forced_align_workspace(B, Tmax, lmax), "ctc_forced_align: workspace too small");
    const AlCfg c = al_config(lmax);
    const size_t smem = al_smem_bytes(c);
    cudaStream_t st = (cudaStream_t)stream;
    auto* bp = (unsigned long long*)workspace;
    if (dtype == LASR_F32)
        launch_align<float>(c, smem, st, B, logits, ld, lse, targets, tgt_len, frames, Tmax, lmax, V, blank, state, frame_logp, score, spans, bp);
    else if (dtype == LASR_BF16)
        launch_align<bf16>(c, smem, st, B, logits, ld, lse, targets, tgt_len, frames, Tmax, lmax, V, blank, state, frame_logp, score, spans, bp);
    else { set_error("ctc_forced_align: bad dtype"); return LASR_ERR_UNSUPPORTED; }
    return check_launch("ctc_forced_align");
}

}  // extern "C"
