// Fused CTC forward-backward + log-softmax backward  (replaces criterions/hybrid_ctc_attn.py:67-75).
//
// Three launches, all on the caller's stream:
//   K_A  ctc_softmax_gather  (all SMs, HBM-bound): one read of the logits, one write of the gradient.
//        per row (t,b): lse = logsumexp(x); grad = s * softmax(x)   (0 and NO read for t >= in_len[b]);
//        lp_ext[b][t][0] = x[blank]-lse, lp_ext[b][t][k+1] = x[label_k]-lse  (compact lattice inputs).
//   K_B  ctc_lattice_warp (grid (B, 2): the alpha sweep and the beta sweep of an utterance run CONCURRENTLY on two CTAs;
//        each thread owns R consecutive state pairs (blank 2k, label 2k+1) in registers, neighbours are registers /
//        one warp shuffle / one shared-memory edge value per warp; L <= 63 labels fit ONE warp -> no barrier at all).
//        The recursion is blank-normalised (a~_t(s) = alpha_t(s) - sum_{tau<=t} lp_tau(blank): |a~| ~ 1e2 instead of
//        T log V ~ 1e4, 10x tighter in fp32) and its inputs are register-prefetched 8 steps ahead.
//   K_C  ctc_scatter_ab (all SMs): occ = exp(alpha + beta - e - tot); grad[t,b,blank] -= s * sum_k occ_blank,
//        grad[t,b,label_k] -= s * occ_label  (red.add; only rows t < in_len[b], only L+1 addresses per row).
// Physical traffic is therefore ~1 read + 1 write of the (T,B,V) tensor plus O(T*B*L) lattice state,
// instead of the ~7 dense passes of log_softmax + ctc_loss + their backward kernels.
#include "common.cuh"

namespace lasr {

// ---------------------------------------------------------------------------------------------
// K_A
// ---------------------------------------------------------------------------------------------
constexpr float LOG2E = 1.4426950408889634f;
constexpr double LN2 = 0.6931471805599453;
// "log zero" of the lattice: a large FINITE sentinel instead of -inf.  max/sub/ex2/lg2 need no guard then (two sentinels
// combine to sentinel + 1 == sentinel in fp32, a sentinel next to a live value contributes ex2(-1e30) = 0), which removes the
// compare/select pair from every log-sum-exp on the sequential critical path.
constexpr float LNEG = -1.0e30f;

template <typename T> struct Vec4;
template <> struct Vec4<float> {
    typedef float4 type;
    static __device__ __forceinline__ void unpack(const float4& v, float* f) { f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w; }
    static __device__ __forceinline__ float4 pack(const float* f) { return make_float4(f[0], f[1], f[2], f[3]); }
};
template <> struct Vec4<bf16> {
    typedef uint2 type;
    static __device__ __forceinline__ void unpack(const uint2& v, float* f) {
        const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&v.x), b = *reinterpret_cast<const __nv_bfloat162*>(&v.y);
        f[0] = __low2float(a); f[1] = __high2float(a); f[2] = __low2float(b); f[3] = __high2float(b);
    }
    static __device__ __forceinline__ uint2 pack(const float* f) {
        __nv_bfloat162 a = __floats2bfloat162_rn(f[0], f[1]), b = __floats2bfloat162_rn(f[2], f[3]);
        uint2 u; u.x = *reinterpret_cast<uint32_t*>(&a); u.y = *reinterpret_cast<uint32_t*>(&b);
        return u;
    }
};

struct CtcDenseParams {
    const void* logits;
    void* grad;
    long st, sb, gst, gsb;
    const int64_t* targets;
    const int64_t* in_len;
    const int64_t* tgt_len;
    float* lp_ext;
    int T, B, V, lmax, blank;
    float grad_scale;
    const float* upstream;
};

// GROUP threads cooperate on one row; each holds NI chunks of 4 consecutive classes in registers.
template <typename T, int GROUP, int NI>
__global__ void __launch_bounds__(256) ctc_softmax_gather_kernel(const CtcDenseParams p) {
    constexpr int ROWS = 256 / GROUP;
    __shared__ float red[ROWS][8];
    const int g = threadIdx.x / GROUP, gl = threadIdx.x % GROUP;
    const long row = (long)blockIdx.x * ROWS + g;
    const bool row_ok = row < (long)p.T * p.B;
    const int t = row_ok ? (int)(row / p.B) : 0, b = row_ok ? (int)(row % p.B) : 0;
    const int Tb = (int)p.in_len[b];
    const bool live = row_ok && t < Tb;
    const T* x = reinterpret_cast<const T*>(p.logits) + (long)t * p.st + (long)b * p.sb;
    T* gout = reinterpret_cast<T*>(p.grad) + (long)t * p.gst + (long)b * p.gsb;
    typedef typename Vec4<T>::type V4;
    float s = p.grad_scale;
    if (p.upstream) s *= __ldg(p.upstream);

    float v[NI][4];
    float mx = -INFINITY;
    if (live) {
#pragma unroll
        for (int i = 0; i < NI; ++i) {
            const int c = (i * GROUP + gl) * 4;
            if (c + 3 < p.V) {
                const V4 raw = *reinterpret_cast<const V4*>(x + c);
                Vec4<T>::unpack(raw, v[i]);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) v[i][j] = (c + j < p.V) ? to_f32<T>(x[c + j]) : -INFINITY;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) mx = fmaxf(mx, v[i][j]);
        }
    }
    // group max
    if (GROUP == 32) {
        mx = warp_max(mx);
    } else {
        mx = warp_max(mx);
        if ((threadIdx.x & 31) == 0) red[0][threadIdx.x >> 5] = mx;
        __syncthreads();
        mx = red[0][0];
#pragma unroll
        for (int w = 1; w < 8; ++w) mx = fmaxf(mx, red[0][w]);
        __syncthreads();
    }
    float sum = 0.f;
    if (live) {
#pragma unroll
        for (int i = 0; i < NI; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                v[i][j] = expf(v[i][j] - mx);  // exp(-inf) = 0 for the padded tail
                sum += v[i][j];
            }
    }
    if (GROUP == 32) {
        sum = warp_sum(sum);
    } else {
        sum = warp_sum(sum);
        if ((threadIdx.x & 31) == 0) red[0][threadIdx.x >> 5] = sum;
        __syncthreads();
        sum = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) sum += red[0][w];
    }
    if (!row_ok) return;
    if (live) {
        const float k = s / sum;
#pragma unroll
        for (int i = 0; i < NI; ++i) {
            const int c = (i * GROUP + gl) * 4;
            float o[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) o[j] = v[i][j] * k;
            if (c + 3 < p.V) {
                *reinterpret_cast<V4*>(gout + c) = Vec4<T>::pack(o);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (c + j < p.V) gout[c + j] = from_f32<T>(o[j]);
            }
        }
        // compact lattice inputs (re-read hits L1/L2: this CTA just streamed the row)
        const float lse = mx + logf(sum);
        const int L = (int)p.tgt_len[b];
        float* le = p.lp_ext + ((long)b * p.T + t) * (p.lmax + 1);
        const int64_t* tg = p.targets + (long)b * p.lmax;
        const float xb = to_f32<T>(x[p.blank]);
        for (int k2 = gl; k2 <= L; k2 += GROUP)  // log2 units: the lattice runs on ex2 / lg2 directly
            le[k2] = LOG2E * ((k2 == 0) ? (xb - lse) : (to_f32<T>(x[(int)tg[k2 - 1]]) - xb));
    } else {
        float z[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int i = 0; i < NI; ++i) {
            const int c = (i * GROUP + gl) * 4;
            if (c + 3 < p.V) {
                *reinterpret_cast<V4*>(gout + c) = Vec4<T>::pack(z);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (c + j < p.V) gout[c + j] = from_f32<T>(0.f);
            }
        }
    }
}

// generic fallback: any V / alignment, one CTA per row, re-reads through L1/L2
template <typename T>
__global__ void __launch_bounds__(256) ctc_softmax_gather_generic(const CtcDenseParams p) {
    __shared__ float scratch[32];
    const long row = blockIdx.x;
    const int t = (int)(row / p.B), b = (int)(row % p.B);
    const int Tb = (int)p.in_len[b];
    const T* x = reinterpret_cast<const T*>(p.logits) + (long)t * p.st + (long)b * p.sb;
    T* gout = reinterpret_cast<T*>(p.grad) + (long)t * p.gst + (long)b * p.gsb;
    if (t >= Tb) {
        for (int c = threadIdx.x; c < p.V; c += 256) gout[c] = from_f32<T>(0.f);
        return;
    }
    float s = p.grad_scale;
    if (p.upstream) s *= __ldg(p.upstream);
    float mx = -INFINITY;
    for (int c = threadIdx.x; c < p.V; c += 256) mx = fmaxf(mx, to_f32<T>(x[c]));
    mx = block_max(mx, scratch);
    float sum = 0.f;
    for (int c = threadIdx.x; c < p.V; c += 256) sum += expf(to_f32<T>(x[c]) - mx);
    sum = block_sum(sum, scratch);
    const float k = s / sum;
    for (int c = threadIdx.x; c < p.V; c += 256) gout[c] = from_f32<T>(expf(to_f32<T>(x[c]) - mx) * k);
    const float lse = mx + logf(sum);
    const int L = (int)p.tgt_len[b];
    float* le = p.lp_ext + ((long)b * p.T + t) * (p.lmax + 1);
    const int64_t* tg = p.targets + (long)b * p.lmax;
    const float xb = to_f32<T>(x[p.blank]);
    for (int k2 = threadIdx.x; k2 <= L; k2 += 256)
        le[k2] = LOG2E * ((k2 == 0) ? (xb - lse) : (to_f32<T>(x[(int)tg[k2 - 1]]) - xb));
}

// ---------------------------------------------------------------------------------------------
// K_B lattice, register-resident.  grid (B, 2): y = 0 runs the alpha sweep, y = 1 the
// beta sweep -- the two recursions are independent, so they run concurrently on different SMs and the occupancy
// exp(alpha + beta - e - tot) is formed by the scatter kernel.  Lane l owns the R consecutive state pairs
// k = l*R .. l*R + R-1 (W = lmax + 1 <= 32 R): inside a lane the neighbour values are registers, across lanes ONE warp
// shuffle per step; there is no shared memory and no block barrier on the critical path, whose length per time step is
// shfl + max + ex2 + add + lg2 (fast intrinsics: their 2^-22 error is below the fp32 ulp of the lattice values).
// Inputs are register-prefetched PF steps ahead.
// ---------------------------------------------------------------------------------------------
// log2-domain log-sum-exp on the raw MUFU ops (ex2.approx.ftz / lg2.approx.ftz: no denormal fix-up code, no scaling by
// log2(e) / ln 2); their 2^-22 relative error is below the fp32 ulp of the lattice values.
__device__ __forceinline__ float fex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float flg2(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// The largest term of a log-sum-exp is exactly 2^0: ordering the inputs with min/max (ALU) saves one MUFU.EX2 per call --
// the lattice step is bound by the MUFU pipe (5 ex2 + 2 lg2 per state pair before, 3 + 2 now).
__device__ __forceinline__ float lse2q(float a, float b) {
    const float m = fmaxf(a, b), lo = fminf(a, b);
    return m + flg2(1.f + fex2(lo - m));
}
__device__ __forceinline__ float lse3q(float a, float b, float c) {
    const float hi = fmaxf(a, b), lo = fminf(a, b);
    const float m = fmaxf(hi, c), mid = fminf(hi, c);
    return m + flg2(1.f + fex2(mid - m) + fex2(lo - m));
}

template <int R, int PFW, int NW>
__global__ void __launch_bounds__(32 * NW) ctc_lattice_warp_kernel(const float* __restrict__ lp_ext, float2* __restrict__ al,
                                                                   float2* __restrict__ be, const int64_t* __restrict__ targets,
                                                                   const int64_t* __restrict__ in_len,
                                                                   const int64_t* __restrict__ tgt_len, float* __restrict__ nll,
                                                                   float* __restrict__ tot_out, int T, int lmax) {
    __shared__ float edge[2][2][NW];  // [parity][value][warp]: boundary states handed to the neighbouring warp (NW > 1)
    __shared__ float fin[2];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool is_beta = blockIdx.y != 0;
    const int Tb = min((int)in_len[b], T), L = min((int)tgt_len[b], lmax);
    const int W = lmax + 1;
    if (Tb <= 0) {
        if (!is_beta && tid == 0) { nll[b] = (L == 0) ? 0.f : INFINITY; tot_out[b] = (L == 0) ? 0.f : -INFINITY; }
        return;
    }
    const int64_t* tg = targets + (long)b * lmax;
    const float* lpb = lp_ext + (long)b * T * W;
    const float NEG = LNEG;
    int kcol[R];          // column of this pair's label emission in lp_ext (clamped: idle pairs read valid memory)
    bool v_lb[R], skip[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int k = tid * R + r;
        kcol[r] = min(k, lmax - 1) + 1;
        v_lb[r] = k < L;
        const long my = (k < L) ? tg[k] : -1;
        if (!is_beta) skip[r] = (k >= 1 && k < L) && (tg[k - 1] != my);   // alpha: 2k-1 -> 2k+1 allowed
        else skip[r] = (k + 1 < L) && (tg[k + 1] != my);                    // beta : 2k+1 -> 2k+3 allowed
    }
    float s_bl[R], s_lb[R];
    float cl[PFW][R], nl[PFW][R];

    if (!is_beta) {
        // C = sum_t lp_t(blank) (double): the normalisation offset of the blank-normalised recursion (see ctc_lattice_kernel)
        double csum = 0.0;
        if (warp == 0) {
            for (int t = lane; t < Tb; t += 32) csum += (double)lpb[(long)t * W];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) csum += __shfl_xor_sync(0xffffffffu, csum, o);
        }
        float2* alb = al + (long)b * T * W;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int k = tid * R + r;
            s_bl[r] = (k == 0) ? 0.f : NEG;
            s_lb[r] = (k == 0 && L > 0) ? lpb[kcol[r]] : NEG;
            if (k < W) alb[k] = make_float2(s_bl[r], s_lb[r]);
        }
        if (NW > 1) {
            if (lane == 31) edge[0][0][warp] = s_lb[R - 1];
            __syncthreads();
        }
#pragma unroll
        for (int i = 0; i < PFW; ++i) {
            const int t = min(1 + i, Tb - 1);
#pragma unroll
            for (int r = 0; r < R; ++r) cl[i][r] = lpb[(long)t * W + kcol[r]];
        }
        for (int t0 = 1; t0 < Tb; t0 += PFW) {
#pragma unroll
            for (int i = 0; i < PFW; ++i) {
                const int t = min(t0 + PFW + i, Tb - 1);
#pragma unroll
                for (int r = 0; r < R; ++r) nl[i][r] = lpb[(long)t * W + kcol[r]];
            }
#pragma unroll
            for (int i = 0; i < PFW; ++i) {
                const int t = t0 + i;
                if (t < Tb) {  // CTA-uniform
                    float up = __shfl_up_sync(0xffffffffu, s_lb[R - 1], 1);
                    if (lane == 0) up = (NW > 1 && warp > 0) ? edge[(t - 1) & 1][0][warp - 1] : NEG;
                    float n_bl[R], n_lb[R];
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const float prev = (r == 0) ? up : s_lb[r - 1];   // alpha_{t-1}(2k-1)
                        n_bl[r] = lse2q(s_bl[r], prev);
                        n_lb[r] = cl[i][r] + lse3q(s_lb[r], s_bl[r], skip[r] ? prev : NEG);
                    }
                    // pairs beyond L need no masking here: alpha only flows towards higher states, so whatever they hold never
                    // reaches a live state (and nothing downstream reads them)
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        s_bl[r] = n_bl[r];
                        s_lb[r] = n_lb[r];
                        const int k = tid * R + r;
                        if (k < W) alb[(long)t * W + k] = make_float2(s_bl[r], s_lb[r]);
                    }
                    if (NW > 1) {
                        if (lane == 31) edge[t & 1][0][warp] = s_lb[R - 1];
                        __syncthreads();
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < PFW; ++i)
#pragma unroll
                for (int r = 0; r < R; ++r) cl[i][r] = nl[i][r];
        }
        if (tid == 0) { fin[0] = NEG; fin[1] = NEG; }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int k = tid * R + r;
            if (k == L) fin[0] = s_bl[r];
            if (L > 0 && k == L - 1) fin[1] = s_lb[r];
        }
        __syncthreads();
        if (tid == 0) {
            const float tot = lse2q(fin[0], fin[1]);          // log2 units, blank-normalised
            const bool feasible = tot > 0.5f * LNEG;
            nll[b] = feasible ? (float)(-((double)tot + csum) * LN2) : INFINITY;
            tot_out[b] = feasible ? tot : -INFINITY;
        }
    } else {
        float2* beb = be + (long)b * T * W;
        {
            const int t = Tb - 1;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int k = tid * R + r;
                const float ld_ = lpb[(long)t * W + kcol[r]];
                s_bl[r] = (k == L) ? 0.f : NEG;
                s_lb[r] = (L > 0 && k == L - 1) ? ld_ : NEG;
                if (k < W) beb[(long)t * W + k] = make_float2(s_bl[r], s_lb[r]);
            }
            if (NW > 1) {
                if (lane == 0) { edge[t & 1][0][warp] = s_bl[0]; edge[t & 1][1][warp] = s_lb[0]; }
                __syncthreads();
            }
        }
#pragma unroll
        for (int i = 0; i < PFW; ++i) {
            const int t = max(Tb - 2 - i, 0);
#pragma unroll
            for (int r = 0; r < R; ++r) cl[i][r] = lpb[(long)t * W + kcol[r]];
        }
        for (int t0 = Tb - 2; t0 >= 0; t0 -= PFW) {
#pragma unroll
            for (int i = 0; i < PFW; ++i) {
                const int t = max(t0 - PFW - i, 0);
#pragma unroll
                for (int r = 0; r < R; ++r) nl[i][r] = lpb[(long)t * W + kcol[r]];
            }
#pragma unroll
            for (int i = 0; i < PFW; ++i) {
                const int t = t0 - i;
                if (t >= 0) {
                    float d1 = __shfl_down_sync(0xffffffffu, s_bl[0], 1);  // beta_{t+1}(2k+2) of the next thread's first pair
                    float d2 = __shfl_down_sync(0xffffffffu, s_lb[0], 1);  // beta_{t+1}(2k+3)
                    if (lane == 31) {
                        const bool has = NW > 1 && warp + 1 < NW;
                        d1 = has ? edge[(t + 1) & 1][0][warp + 1] : NEG;
                        d2 = has ? edge[(t + 1) & 1][1][warp + 1] : NEG;
                    }
                    float n_bl[R], n_lb[R];
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const float x1 = (r == R - 1) ? d1 : s_bl[r + 1];
                        const float x2 = (r == R - 1) ? d2 : s_lb[r + 1];
                        n_bl[r] = lse2q(s_bl[r], s_lb[r]);
                        n_lb[r] = cl[i][r] + lse3q(s_lb[r], x1, skip[r] ? x2 : NEG);
                    }
                    // dead blank states stay at the sentinel by themselves (sentinel + lg2(2) == sentinel); dead LABEL states must be
                    // forced: their emission column was never written by the gather kernel (k > L), and beta flows downwards
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        s_bl[r] = n_bl[r];
                        s_lb[r] = v_lb[r] ? n_lb[r] : NEG;
                        const int k = tid * R + r;
                        if (k < W) beb[(long)t * W + k] = make_float2(s_bl[r], s_lb[r]);
                    }
                    if (NW > 1) {
                        if (lane == 0) { edge[t & 1][0][warp] = s_bl[0]; edge[t & 1][1][warp] = s_lb[0]; }
                        __syncthreads();
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < PFW; ++i)
#pragma unroll
                for (int r = 0; r < R; ++r) cl[i][r] = nl[i][r];
        }
    }
}

// scatter for the split lattice: occupancy formed on the fly from alpha, beta, the label emission term and tot
template <typename GT>
__global__ void __launch_bounds__(256) ctc_scatter_ab_kernel(const float2* __restrict__ al, const float2* __restrict__ be,
                                                             const float* __restrict__ lp_ext, const float* __restrict__ tot,
                                                             void* grad, long gst, long gsb, const int64_t* __restrict__ targets,
                                                             const int64_t* __restrict__ in_len,
                                                             const int64_t* __restrict__ tgt_len, int T, int B, int lmax,
                                                             int blank, float grad_scale, const float* upstream) {
    const long row = (long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= (long)T * B) return;
    const int lane = threadIdx.x & 31;
    const int t = (int)(row / B), b = (int)(row % B);
    if (t >= (int)in_len[b]) return;
    const int L = min((int)tgt_len[b], lmax), W = lmax + 1;
    float s = grad_scale;
    if (upstream) s *= __ldg(upstream);
    const long base = ((long)b * T + t) * W;
    const float tt = tot[b];
    const bool feasible = tt > -INFINITY;
    const float qnan = __int_as_float(0x7fc00000);
    const int64_t* tg = targets + (long)b * lmax;
    GT* g = reinterpret_cast<GT*>(grad) + (long)t * gst + (long)b * gsb;
    float bsum = 0.f;
    for (int k = lane; k <= L; k += 32) {
        const float2 a = al[base + k], bb = be[base + k];
        float o_bl = fex2(a.x + bb.x - tt);              // log2 units; a sentinel on either side gives ex2(-1e30) = 0
        if (!feasible) o_bl = qnan;
        bsum += o_bl;
        if (k < L) {
            const float e = lp_ext[base + k + 1];
            float o_lb = fex2(a.y + bb.y - e - tt);
            if (!feasible) o_lb = qnan;
            const int c = (int)tg[k];
            if constexpr (sizeof(GT) == 4) atomicAdd(reinterpret_cast<float*>(g) + c, -s * o_lb);
            else atomicAdd(reinterpret_cast<bf16*>(g) + c, __float2bfloat16_rn(-s * o_lb));
        }
    }
    bsum = warp_sum(bsum);
    if (lane == 0) {
        if constexpr (sizeof(GT) == 4) atomicAdd(reinterpret_cast<float*>(g) + blank, -s * bsum);
        else atomicAdd(reinterpret_cast<bf16*>(g) + blank, __float2bfloat16_rn(-s * bsum));
    }
}

template <typename T>
static int ctc_launch(const CtcDenseParams& p, float2* ab, float2* be, float* tot, float* nll, cudaStream_t st) {
    const long rows = (long)p.T * p.B;
    const bool vec = ((reinterpret_cast<uintptr_t>(p.logits) | reinterpret_cast<uintptr_t>(p.grad)) % (4 * sizeof(T)) == 0) &&
                     p.st % 4 == 0 && p.sb % 4 == 0 && p.gst % 4 == 0 && p.gsb % 4 == 0;
    bool done = false;
    if (vec) {
        const int chunks = (p.V + 3) / 4;
#define LASR_CTC_CASE(GROUP, NI)                                                                        \
    if (!done && chunks <= GROUP * NI) {                                                                \
        ctc_softmax_gather_kernel<T, GROUP, NI><<<ceil_div(rows, 256 / GROUP), 256, 0, st>>>(p);         \
        done = true;                                                                                    \
    }
        LASR_CTC_CASE(32, 1) LASR_CTC_CASE(32, 2) LASR_CTC_CASE(32, 4) LASR_CTC_CASE(32, 8)
        LASR_CTC_CASE(256, 2) LASR_CTC_CASE(256, 4) LASR_CTC_CASE(256, 6) LASR_CTC_CASE(256, 8)
#undef LASR_CTC_CASE
    }
    if (!done) ctc_softmax_gather_generic<T><<<(unsigned)rows, 256, 0, st>>>(p);
    int rc = check_launch("ctc_softmax_gather");
    if (rc) return rc;
    // R state pairs per thread, NW warps per sweep (32 R NW >= W)
    const int W = p.lmax + 1;
    dim3 grid(p.B, 2);
#define LASR_LATTICE(R, PFW, NW) \
    ctc_lattice_warp_kernel<R, PFW, NW><<<grid, 32 * NW, 0, st>>>(p.lp_ext, ab, be, p.targets, p.in_len, p.tgt_len, nll, tot, p.T, p.lmax)
    if (W <= 32) LASR_LATTICE(1, 8, 1);
    else if (W <= 64) LASR_LATTICE(2, 8, 1);
    else if (W <= 128) LASR_LATTICE(2, 8, 2);
    else if (W <= 256) LASR_LATTICE(2, 8, 4);
    else if (W <= 512) LASR_LATTICE(2, 8, 8);
    else LASR_LATTICE(4, 4, 8);
#undef LASR_LATTICE
    rc = check_launch("ctc_lattice_warp");
    if (rc) return rc;
    ctc_scatter_ab_kernel<T><<<ceil_div(rows, 8), 256, 0, st>>>(ab, be, p.lp_ext, tot, p.grad, p.gst, p.gsb, p.targets, p.in_len,
                                                               p.tgt_len, p.T, p.B, p.lmax, p.blank, p.grad_scale, p.upstream);
    return check_launch("ctc_scatter_ab");
}

}  // namespace lasr

extern "C" {

size_t lasr_ctc_workspace_bytes(int T, int B, int lmax) {
    const size_t w = (size_t)(lmax < 1 ? 1 : lmax) + 1;
    // alpha (float2) + beta (float2) + gathered lattice inputs (float) per (t, b, state pair); tot per utterance
    return (size_t)T * B * w * (sizeof(float) + 2 * sizeof(float2)) + (size_t)B * sizeof(float) + 1024;
}

int lasr_ctc_fwdbwd(const void* logits, int dtype, int64_t st, int64_t sb, const int64_t* targets, const int64_t* in_len,
                    const int64_t* tgt_len, int T, int B, int V, int lmax, int blank, float grad_scale,
                    const float* upstream, float* nll, void* grad, int64_t gst, int64_t gsb, void* workspace,
                    size_t ws_bytes, void* stream) {
    using namespace lasr;
    LASR_REQUIRE(logits && targets && in_len && tgt_len && nll && grad && workspace, "ctc: null pointer");
    LASR_REQUIRE(T > 0 && B > 0 && V > 1 && lmax >= 1, "ctc: bad shape T=%d B=%d V=%d lmax=%d", T, B, V, lmax);
    LASR_REQUIRE(lmax + 1 <= 1024, "ctc: lmax=%d exceeds the 1023-label lattice CTA", lmax);
    LASR_REQUIRE(blank >= 0 && blank < V, "ctc: bad blank");
    LASR_REQUIRE(ws_bytes >= lasr_ctc_workspace_bytes(T, B, lmax), "ctc: workspace too small");
    CtcDenseParams p;
    p.logits = logits; p.grad = grad; p.st = st; p.sb = sb; p.gst = gst; p.gsb = gsb;
    p.targets = targets; p.in_len = in_len; p.tgt_len = tgt_len;
    const size_t w = (size_t)lmax + 1;
    uintptr_t base = (reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255;
    float2* ab = reinterpret_cast<float2*>(base);
    float2* be = reinterpret_cast<float2*>(base + (size_t)T * B * w * sizeof(float2));
    p.lp_ext = reinterpret_cast<float*>(base + 2 * (size_t)T * B * w * sizeof(float2));
    float* tot = reinterpret_cast<float*>(base + (size_t)T * B * w * (2 * sizeof(float2) + sizeof(float)));
    p.T = T; p.B = B; p.V = V; p.lmax = lmax; p.blank = blank; p.grad_scale = grad_scale; p.upstream = upstream;
    if (dtype == LASR_F32) return ctc_launch<float>(p, ab, be, tot, nll, (cudaStream_t)stream);
    if (dtype == LASR_BF16) return ctc_launch<bf16>(p, ab, be, tot, nll, (cudaStream_t)stream);
    set_error("ctc: unsupported dtype %d", dtype);
    return LASR_ERR_UNSUPPORTED;
}

}  // extern "C"
