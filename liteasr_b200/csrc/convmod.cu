// Conformer convolution-module middle (nets/conformer_convolution.py:49-53 and its backward):
//   GLU -> depthwise Conv1d(k=15, pad 7, groups=d) -> BatchNorm1d (train: batch stats over ALL B*T'
//   frames, padding included -- quirk Q2) -> Swish.
// Layout is (B, T', C) with channels contiguous (what the GEMMs produce/consume), so the reference's
// transposes vanish and every access is coalesced over channels.
// Fast kernels (d % 4 == 0): one CTA per (32-step time chunk, utterance, 128-channel block).  Phase 1 stages the
// 46-row halo tile in shared memory with 64/128-bit loads (all loads of a CTA in flight at once), applying the
// pointwise math (GLU; BatchNorm + Swish backward) on the way in; phase 2 gives each thread one channel pair and
// 8 time steps and slides the 15-tap window through registers (static indexing, conflict-free float2 LDS).
// The *_generic kernels (any even d) keep the register-window-only scheme.
//   fwd 1: z = dwconv(glu(y2)) + per-(batch,chunk) partial sum / sum-of-squares   (deterministic)
//   fwd 2: finalize stats (double), running-stat update (momentum 0.1, unbiased var)
//   fwd 3: a = swish(gamma * (z - mean) * rstd + beta)
//   bwd 1: partial sums of du and du*zhat  (du = da * swish'(u))  -> also dgamma / dbeta
//   bwd 2: dz on the fly -> depthwise dgrad + wgrad -> GLU backward, one pass
#include <cooperative_groups.h>

#include "common.cuh"

namespace lasr {

constexpr int KW = 15, HALO = 7, TCH = 32;
constexpr int NRED = KW + 3;  // depthwise taps + bias + the two pointwise-bias column sums

template <typename TD> __device__ __forceinline__ float2 ld2(const TD* p);
template <> __device__ __forceinline__ float2 ld2<float>(const float* p) { return *reinterpret_cast<const float2*>(p); }
template <> __device__ __forceinline__ float2 ld2<bf16>(const bf16* p) {
    const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(p);
    return make_float2(__low2float(h), __high2float(h));
}
template <typename TD> __device__ __forceinline__ void st2(TD* p, float a, float b);
template <> __device__ __forceinline__ void st2<float>(float* p, float a, float b) { *reinterpret_cast<float2*>(p) = make_float2(a, b); }
template <> __device__ __forceinline__ void st2<bf16>(bf16* p, float a, float b) {
    *reinterpret_cast<__nv_bfloat162*>(p) = __floats2bfloat162_rn(a, b);
}

// ---------------------------------------------------------------- fwd 1
// LENS (lasr_glu_dwconv_fwd_lens): GLU outputs of rows t >= lens[b] read as zero -- the Conv1d zero padding the batch-1 call on
// the utterance cut to lens[b] frames sees -- so that rows t < lens[b] do not depend on the padded rows.
__device__ __forceinline__ int valid_rows(const int64_t* lens, int b, int T) {
    const long l = lens[b];
    return (int)(l < T ? (l < 0 ? 0 : l) : T);
}

template <typename TD, bool LENS = false>
__global__ void __launch_bounds__(128) glu_dwconv_fwd_generic(const TD* __restrict__ y2, long ldy, const float* __restrict__ w,
                                                             const float* __restrict__ bias, float* __restrict__ z,
                                                             float* __restrict__ partial, int T, int d, const int64_t* __restrict__ lens) {
    const int b = blockIdx.y, chunk = blockIdx.x, nchunk = gridDim.x;
    const int Tv = LENS ? valid_rows(lens, b, T) : T;
    const int t0 = chunk * TCH, t1 = min(T, t0 + TCH);
    float* part = partial + ((long)(b * nchunk + chunk)) * 2 * d;
    for (int c = threadIdx.x * 2; c < d; c += blockDim.x * 2) {
        float w0[KW], w1[KW], r0[KW], r1[KW];
#pragma unroll
        for (int k = 0; k < KW; ++k) { w0[k] = w[c * KW + k]; w1[k] = w[(c + 1) * KW + k]; r0[k] = 0.f; r1[k] = 0.f; }
        const float b0 = bias[c], b1 = bias[c + 1];
        float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
        for (int tt = t0 - HALO; tt < t1 + HALO; ++tt) {
            float g0 = 0.f, g1 = 0.f;
            if (tt >= 0 && tt < Tv) {
                const TD* row = y2 + ((long)b * T + tt) * ldy;
                const float2 v = ld2<TD>(row + c), gt = ld2<TD>(row + d + c);
                g0 = v.x * sigmoidf_(gt.x);
                g1 = v.y * sigmoidf_(gt.y);
            }
#pragma unroll
            for (int k = 0; k < KW - 1; ++k) { r0[k] = r0[k + 1]; r1[k] = r1[k + 1]; }
            r0[KW - 1] = g0; r1[KW - 1] = g1;
            const int t = tt - HALO;  // window now holds g[t-7 .. t+7]
            if (t >= t0) {
                float a0 = b0, a1 = b1;
#pragma unroll
                for (int k = 0; k < KW; ++k) { a0 = fmaf(w0[k], r0[k], a0); a1 = fmaf(w1[k], r1[k], a1); }
                *reinterpret_cast<float2*>(z + ((long)b * T + t) * d + c) = make_float2(a0, a1);
                s0 += a0; s1 += a1; q0 += a0 * a0; q1 += a1 * a1;
            }
        }
        part[c] = s0; part[c + 1] = s1;
        part[d + c] = q0; part[d + c + 1] = q1;
    }
}

// ---------------------------------------------------------------- fwd 3
template <typename TD>
__global__ void __launch_bounds__(256) bn_swish_fwd_kernel(const float* __restrict__ z, const float* __restrict__ mean,
                                                           const float* __restrict__ rstd, const float* __restrict__ gamma,
                                                           const float* __restrict__ beta, TD* __restrict__ a, long n, int d) {
    const long i = ((long)blockIdx.x * 256 + threadIdx.x) * 2;
    if (i >= n) return;
    const int c = (int)(i % d);
    const float2 v = *reinterpret_cast<const float2*>(z + i);
    const float u0 = (v.x - mean[c]) * rstd[c] * gamma[c] + beta[c];
    const float u1 = (v.y - mean[c + 1]) * rstd[c + 1] * gamma[c + 1] + beta[c + 1];
    st2<TD>(a + i, swishf_(u0), swishf_(u1));
}

// d % 4 == 0: one thread = 4 channels x 4 rows (rows strided by the grid), per-channel scale/shift folded once
template <typename TD>
__global__ void __launch_bounds__(256) bn_swish_fwd_vec_kernel(const float* __restrict__ z, const float* __restrict__ mean,
                                                               const float* __restrict__ rstd, const float* __restrict__ gamma,
                                                               const float* __restrict__ beta, TD* __restrict__ a, long rows, int d) {
    LASR_PDL_SYNC();
    const int vpr = d >> 2;
    const long gid = (long)blockIdx.x * 256 + threadIdx.x;
    const int cv = (int)(gid % vpr);
    const long r0 = (gid / vpr) * 4;
    if (r0 >= rows) return;
    const int c = cv * 4;
    const float4 m = *reinterpret_cast<const float4*>(mean + c), rs = *reinterpret_cast<const float4*>(rstd + c);
    const float4 ga = *reinterpret_cast<const float4*>(gamma + c), be = *reinterpret_cast<const float4*>(beta + c);
    const float4 sc = make_float4(rs.x * ga.x, rs.y * ga.y, rs.z * ga.z, rs.w * ga.w);
    float4 v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j)
        if (r0 + j < rows) v[j] = *reinterpret_cast<const float4*>(z + (r0 + j) * d + c);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (r0 + j >= rows) break;
        const float u0 = (v[j].x - m.x) * sc.x + be.x, u1 = (v[j].y - m.y) * sc.y + be.y;
        const float u2 = (v[j].z - m.z) * sc.z + be.z, u3 = (v[j].w - m.w) * sc.w + be.w;
        TD* o = a + (r0 + j) * d + c;
        st2<TD>(o, swishf_(u0), swishf_(u1));
        st2<TD>(o + 2, swishf_(u2), swishf_(u3));
    }
}

// ---------------------------------------------------------------- bwd 1
template <typename TD>
__global__ void __launch_bounds__(128) bn_swish_bwd_stats_generic(const TD* __restrict__ da, const float* __restrict__ z,
                                                                 const float* __restrict__ mean, const float* __restrict__ rstd,
                                                                 const float* __restrict__ gamma, const float* __restrict__ beta,
                                                                 float* __restrict__ partial, long rows, int d) {
    const long r0 = (long)blockIdx.x * TCH, r1 = min(rows, r0 + TCH);
    float* part = partial + (long)blockIdx.x * 2 * d;
    for (int c = threadIdx.x * 2; c < d; c += blockDim.x * 2) {
        const float m0 = mean[c], m1 = mean[c + 1], rs0 = rstd[c], rs1 = rstd[c + 1];
        const float g0 = gamma[c], g1 = gamma[c + 1], be0 = beta[c], be1 = beta[c + 1];
        float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
        for (long r = r0; r < r1; ++r) {
            const float2 zz = *reinterpret_cast<const float2*>(z + r * d + c);
            const float2 g = ld2<TD>(da + r * d + c);
            const float zh0 = (zz.x - m0) * rs0, zh1 = (zz.y - m1) * rs1;
            const float du0 = g.x * dswishf_(g0 * zh0 + be0), du1 = g.y * dswishf_(g1 * zh1 + be1);
            s0 += du0; s1 += du1; q0 += du0 * zh0; q1 += du1 * zh1;
        }
        part[c] = s0; part[c + 1] = s1;
        part[d + c] = q0; part[d + c + 1] = q1;
    }
}

// ---------------------------------------------------------------- bwd 2
template <typename TD>
__global__ void __launch_bounds__(128) dwconv_glu_bwd_generic(const TD* __restrict__ da, const float* __restrict__ z,
                                                             const TD* __restrict__ y2, long ldy, const float* __restrict__ mean,
                                                             const float* __restrict__ rstd, const float* __restrict__ gamma,
                                                             const float* __restrict__ beta, const float* __restrict__ sums,
                                                             const float* __restrict__ w, TD* __restrict__ dy2, long lddy,
                                                             float* __restrict__ dw, float* __restrict__ dbias, int T, int d,
                                                             float inv_count) {
    const int b = blockIdx.y, t0 = blockIdx.x * TCH, t1 = min(T, t0 + TCH);
    for (int c = threadIdx.x * 2; c < d; c += blockDim.x * 2) {
        float w0[KW], w1[KW], z0[KW], z1[KW], g0r[KW], g1r[KW], aw0[KW], aw1[KW];
#pragma unroll
        for (int k = 0; k < KW; ++k) {
            w0[k] = w[c * KW + k]; w1[k] = w[(c + 1) * KW + k];
            z0[k] = z1[k] = g0r[k] = g1r[k] = aw0[k] = aw1[k] = 0.f;
        }
        const float m0 = mean[c], m1 = mean[c + 1], rs0 = rstd[c], rs1 = rstd[c + 1];
        const float ga0 = gamma[c], ga1 = gamma[c + 1], be0 = beta[c], be1 = beta[c + 1];
        const float ms0 = sums[c] * inv_count, ms1 = sums[c + 1] * inv_count;          // mean(du)
        const float mq0 = sums[d + c] * inv_count, mq1 = sums[d + c + 1] * inv_count;  // mean(du * zhat)
        float ab0 = 0.f, ab1 = 0.f;
        for (int tt = t0 - HALO; tt < t1 + HALO; ++tt) {
            float dz0 = 0.f, dz1 = 0.f, g0 = 0.f, g1 = 0.f;
            if (tt >= 0 && tt < T) {
                const long r = (long)b * T + tt;
                const float2 zz = *reinterpret_cast<const float2*>(z + r * d + c);
                const float2 gd = ld2<TD>(da + r * d + c);
                const float zh0 = (zz.x - m0) * rs0, zh1 = (zz.y - m1) * rs1;
                const float du0 = gd.x * dswishf_(ga0 * zh0 + be0), du1 = gd.y * dswishf_(ga1 * zh1 + be1);
                dz0 = ga0 * rs0 * (du0 - ms0 - zh0 * mq0);
                dz1 = ga1 * rs1 * (du1 - ms1 - zh1 * mq1);
                const TD* row = y2 + r * ldy;
                const float2 v = ld2<TD>(row + c), gt = ld2<TD>(row + d + c);
                g0 = v.x * sigmoidf_(gt.x);
                g1 = v.y * sigmoidf_(gt.y);
            }
#pragma unroll
            for (int k = 0; k < KW - 1; ++k) { z0[k] = z0[k + 1]; z1[k] = z1[k + 1]; g0r[k] = g0r[k + 1]; g1r[k] = g1r[k + 1]; }
            z0[KW - 1] = dz0; z1[KW - 1] = dz1; g0r[KW - 1] = g0; g1r[KW - 1] = g1;
            const int t = tt - HALO;  // windows hold dz / g at times t-7 .. t+7 (index j <-> t-7+j)
            if (t >= t0) {
                // z[t'] = sum_k w[k] g[t'+k-7]  =>  dg[t] = sum_k w[k] dz[t-k+7] (index 14-k)
                float dg0 = 0.f, dg1 = 0.f;
#pragma unroll
                for (int k = 0; k < KW; ++k) { dg0 = fmaf(w0[k], z0[KW - 1 - k], dg0); dg1 = fmaf(w1[k], z1[KW - 1 - k], dg1); }
                // dw[k] += dz[t] * g[t+k-7] ; db += dz[t]
                const float c0 = z0[HALO], c1 = z1[HALO];
#pragma unroll
                for (int k = 0; k < KW; ++k) { aw0[k] = fmaf(c0, g0r[k], aw0[k]); aw1[k] = fmaf(c1, g1r[k], aw1[k]); }
                ab0 += c0; ab1 += c1;
                // GLU backward at t
                const long r = (long)b * T + t;
                const TD* row = y2 + r * ldy;
                const float2 v = ld2<TD>(row + c), gt = ld2<TD>(row + d + c);
                const float sg0 = sigmoidf_(gt.x), sg1 = sigmoidf_(gt.y);
                TD* orow = dy2 + r * lddy;
                st2<TD>(orow + c, dg0 * sg0, dg1 * sg1);
                st2<TD>(orow + d + c, dg0 * v.x * sg0 * (1.f - sg0), dg1 * v.y * sg1 * (1.f - sg1));
            }
        }
#pragma unroll
        for (int k = 0; k < KW; ++k) { atomicAdd(dw + c * KW + k, aw0[k]); atomicAdd(dw + (c + 1) * KW + k, aw1[k]); }
        atomicAdd(dbias + c, ab0);
        atomicAdd(dbias + c + 1, ab1);
    }
}


// =================================================================================================
// fast kernels
// =================================================================================================
// Tile = FT time steps x FC channels per CTA of 256 threads; thread = ONE channel x FT/4 consecutive time steps, so the
// register window is FT/4 + 14 floats + 15 taps (~64 registers -> 4 CTAs / 1024 threads per SM) and every shared-memory /
// global access of a warp covers 32 consecutive channels (conflict-free LDS.32, 128-byte coalesced stores).
constexpr int FT = 64, FC = 64, FWIN = FT + 2 * HALO, FQ = FT / 4;

template <typename TD> __device__ __forceinline__ float4 ld4c(const TD* p);
template <> __device__ __forceinline__ float4 ld4c<float>(const float* p) { return *reinterpret_cast<const float4*>(p); }
template <> __device__ __forceinline__ float4 ld4c<bf16>(const bf16* p) {
    const uint2 u = *reinterpret_cast<const uint2*>(p);
    const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&u.x), b = *reinterpret_cast<const __nv_bfloat162*>(&u.y);
    return make_float4(__low2float(a), __high2float(a), __low2float(b), __high2float(b));
}

// ---------------------------------------------------------------- fwd 1 (fast)
// partial rows keep the 32-step granularity of the ABI: a CTA writes one row per 32-step half of its tile.
template <typename TD, bool LENS = false>
__global__ void __launch_bounds__(256, 4) glu_dwconv_fwd_kernel(const TD* __restrict__ y2, long ldy, const float* __restrict__ w,
                                                                const float* __restrict__ bias, float* __restrict__ z,
                                                                float* __restrict__ partial, int T, int d, const int64_t* __restrict__ lens) {
    LASR_PDL_SYNC();
    __shared__ __align__(16) float gt[FWIN][FC];
    __shared__ float wt[FC * KW];
    __shared__ float red[2][4][FC];
    const int b = blockIdx.y, c0 = blockIdx.z * FC, t0 = blockIdx.x * FT;
    for (int i = threadIdx.x; i < FC * KW; i += 256) wt[i] = (c0 + i / KW < d) ? w[(long)c0 * KW + i] : 0.f;
    // phase 1: GLU of the halo window; a thread's items share the channel quad, all its loads are issued before the math
    {
        const int cv = (threadIdx.x & 15) * 4, rbase = threadIdx.x >> 4;
        constexpr int NIT = (FWIN + 15) / 16;
        float4 v[NIT], gate[NIT];
        const bool cok = c0 + cv < d;
#pragma unroll
        for (int it = 0; it < NIT; ++it) {
            const int r = rbase + 16 * it, tt = t0 - HALO + r;
            v[it] = make_float4(0.f, 0.f, 0.f, 0.f);
            gate[it] = v[it];
            if (r < FWIN && tt >= 0 && tt < (LENS ? valid_rows(lens, b, T) : T) && cok) {
                const TD* row = y2 + ((long)b * T + tt) * ldy + c0 + cv;
                v[it] = ld4c<TD>(row);
                gate[it] = ld4c<TD>(row + d);
            }
        }
#pragma unroll
        for (int it = 0; it < NIT; ++it) {
            const int r = rbase + 16 * it;
            if (r < FWIN)
                *reinterpret_cast<float4*>(&gt[r][cv]) = make_float4(v[it].x * sigmoidf_(gate[it].x), v[it].y * sigmoidf_(gate[it].y),
                                                                    v[it].z * sigmoidf_(gate[it].z), v[it].w * sigmoidf_(gate[it].w));
        }
    }
    __syncthreads();
    const int c = threadIdx.x & (FC - 1), qtr = threadIdx.x >> 6, cg = c0 + c;
    float s = 0.f, q = 0.f;
    if (cg < d) {
        float wk[KW];
#pragma unroll
        for (int k = 0; k < KW; ++k) wk[k] = wt[c * KW + k];
        const float b0 = bias[cg];
        const int tb = qtr * FQ;
        float win[FQ + KW - 1];
#pragma unroll
        for (int j = 0; j < FQ + KW - 1; ++j) win[j] = gt[tb + j][c];
        float* zp = z + ((long)b * T + t0 + tb) * d + cg;
#pragma unroll
        for (int i = 0; i < FQ; ++i) {
            if (t0 + tb + i < T) {
                float a = b0;
#pragma unroll
                for (int k = 0; k < KW; ++k) a = fmaf(wk[k], win[i + k], a);
                zp[(long)i * d] = a;
                s += a;
                q += a * a;
            }
        }
    }
    red[0][qtr][c] = s;
    red[1][qtr][c] = q;
    __syncthreads();
    if (threadIdx.x < 2 * FC) {  // thread -> (half, channel): quarters {0,1} are the first 32 steps, {2,3} the second
        const int half = threadIdx.x >> 6, cc = threadIdx.x & (FC - 1);
        const int n32 = (T + TCH - 1) / TCH, row32 = blockIdx.x * 2 + half;
        if (row32 < n32 && c0 + cc < d) {
            float* part = partial + ((long)b * n32 + row32) * 2 * d;
            part[c0 + cc] = red[0][2 * half][cc] + red[0][2 * half + 1][cc];
            part[d + c0 + cc] = red[1][2 * half][cc] + red[1][2 * half + 1][cc];
        }
    }
}

// ---------------------------------------------------------------- fwd 1 (streaming, bf16, d % 64 == 0)
// One CTA = one utterance x 64 channels, streaming the T' frames in 32-row chunks: no halo re-reads, no tile quantisation at
// T' = 299, and -- the point -- the loads of chunk j + 2 (cp.async, 16 B per thread and tensor half) are in flight while chunk j is
// computed.  The tiled kernel above alternates a load phase and a compute phase per CTA and is ~60 % issue-bound by ~1000
// instructions per thread (ncu: 21.7 M warp instructions, 38 us at C2 / B = 126, 2 TB/s).
//   raw ring (3 stages)  : the value / gate halves of a chunk as they sit in memory; every thread converts exactly the 16 bytes it
//                          fetched itself (no barrier between the copy and the GLU)
//   g ring (64 rows)     : GLU outputs, fp32; chunk j occupies rows [32 j, 32 j + 32) mod 64, so the 14 rows of history a chunk needs
//                          are still there
//   outputs lag 7 rows   : iteration j writes z rows [32 j - 7, 32 j + 25) from g rows [32 j - 14, 32 j + 32); one extra iteration
//                          flushes the tail against zero rows
// Statistics: per-thread running sums over the whole utterance, reduced over the four row groups at the end and written as ONE
// partial row per (utterance, channel block); the utterance's other rows of the ABI's 32-step layout are zeroed.
constexpr int SR = 32, SCH = 64, SRING = 64, SSTG = 3;

__device__ __forceinline__ void cp_async16(void* dst, const void* src, bool valid) {
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst);
    const int n = valid ? 16 : 0;  // src-size 0: the 16 bytes are zero-filled, nothing is read
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(src), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
// sigmoid(x) = 0.5 tanh(x / 2) + 0.5: one MUFU op instead of ex2 + rcp (rel. error ~2^-11, the inputs are bf16)
__device__ __forceinline__ float sigmoid_tanh(float x) {
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.5f * x));
    return fmaf(t, 0.5f, 0.5f);
}
__device__ __forceinline__ uint32_t pack_bf2(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float bf16lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16hi(uint32_t u) { return __uint_as_float(u & 0xffff0000u); }

template <bool LENS = false>
__global__ void __launch_bounds__(256, 4) glu_dwconv_fwd_stream_kernel(const bf16* __restrict__ y2, long ldy, const float* __restrict__ w,
                                                                       const float* __restrict__ bias, float* __restrict__ z,
                                                                       float* __restrict__ partial, int T, int d, const int64_t* __restrict__ lens) {
    LASR_PDL_SYNC();
    __shared__ __align__(16) bf16 raw[SSTG][2][SR][SCH];
    __shared__ __align__(16) float ring[SRING][SCH];
    __shared__ float wt[SCH * KW];
    __shared__ float red[2][4][SCH];
    const int b = blockIdx.y, c0 = blockIdx.x * SCH, tid = threadIdx.x;
    const int nch = (T + SR - 1) / SR;
    const int Tv = LENS ? valid_rows(lens, b, T) : T;
    const int lrow = tid >> 3, lpc = (tid & 7) * 8;     // loader / GLU role: one row, 8 channels
    const int c = tid & (SCH - 1), rg = tid >> 6;       // convolution role: one channel, 8 rows
    const bf16* src0 = y2 + (long)b * T * ldy + c0 + lpc;
    auto issue = [&](int j) {
        const int t = j * SR + lrow;
        const bool ok = j < nch && t < Tv;
        const bf16* sp = src0 + (long)(ok ? t : 0) * ldy;
        cp_async16(&raw[j % SSTG][0][lrow][lpc], sp, ok);
        cp_async16(&raw[j % SSTG][1][lrow][lpc], sp + d, ok);
        cp_async_commit();
    };
    issue(0);
    issue(1);
    for (int i = tid; i < SCH * KW; i += 256) wt[i] = w[(long)c0 * KW + i];
    for (int i = tid; i < SRING * SCH / 4; i += 256) reinterpret_cast<float4*>(&ring[0][0])[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncthreads();
    float wk[KW];
#pragma unroll
    for (int k = 0; k < KW; ++k) wk[k] = wt[c * KW + k];
    const float b0 = bias[c0 + c];
    float s = 0.f, q = 0.f;
    float* zc = z + (long)b * T * d + c0 + c;
    for (int j = 0; j <= nch; ++j) {
        issue(j + 2);
        cp_async_wait<2>();  // this thread's copies of chunk j have landed
        const uint4 v = *reinterpret_cast<const uint4*>(&raw[j % SSTG][0][lrow][lpc]);
        const uint4 gt = *reinterpret_cast<const uint4*>(&raw[j % SSTG][1][lrow][lpc]);
        float4 g0, g1;
        g0.x = bf16lo(v.x) * sigmoid_tanh(bf16lo(gt.x)); g0.y = bf16hi(v.x) * sigmoid_tanh(bf16hi(gt.x));
        g0.z = bf16lo(v.y) * sigmoid_tanh(bf16lo(gt.y)); g0.w = bf16hi(v.y) * sigmoid_tanh(bf16hi(gt.y));
        g1.x = bf16lo(v.z) * sigmoid_tanh(bf16lo(gt.z)); g1.y = bf16hi(v.z) * sigmoid_tanh(bf16hi(gt.z));
        g1.z = bf16lo(v.w) * sigmoid_tanh(bf16lo(gt.w)); g1.w = bf16hi(v.w) * sigmoid_tanh(bf16hi(gt.w));
        __syncthreads();  // the previous iteration's convolution has read the rows this chunk overwrites
        float* rp = &ring[(j * SR + lrow) & (SRING - 1)][lpc];
        *reinterpret_cast<float4*>(rp) = g0;
        *reinterpret_cast<float4*>(rp + 4) = g1;
        __syncthreads();
        const int base = j * SR - 2 * HALO + 8 * rg;  // window row 0; output row i of this thread = base + HALO + i
        float win[8 + KW - 1];
#pragma unroll
        for (int k = 0; k < 8 + KW - 1; ++k) win[k] = ring[(base + k) & (SRING - 1)][c];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int t = base + HALO + i;
            if (t >= 0 && t < T) {
                float a = b0;
#pragma unroll
                for (int k = 0; k < KW; ++k) a = fmaf(wk[k], win[i + k], a);
                zc[(long)t * d] = a;
                s += a;
                q = fmaf(a, a, q);
            }
        }
    }
    cp_async_wait<0>();
    red[0][rg][c] = s;
    red[1][rg][c] = q;
    __syncthreads();
    if (tid < 2 * SCH) {
        const int which = tid >> 6, cc = tid & (SCH - 1);
        const float v = (red[which][0][cc] + red[which][1][cc]) + (red[which][2][cc] + red[which][3][cc]);
        float* part = partial + (long)b * nch * 2 * d + which * d + c0 + cc;
        part[0] = v;
        for (int r = 1; r < nch; ++r) part[(long)r * 2 * d] = 0.f;
    }
}

// ---------------------------------------------------------------- column reduction of [nblk][2][d] partials (double)
// One thread-block CLUSTER of CL CTAs per 32 channels: every CTA (32 channels x RG row groups = 1024 threads) reduces a
// 1/CL slice of the rows, rank 0 then adds the CL slice sums through distributed shared memory in a fixed order
// (deterministic; no global scratch, no atomics).  The reduction is a latency chain per thread, so it is spread over as many
// threads as possible: 8 CTAs x 1024 threads per 32 channels instead of one CTA of 256.
// FIN = 0: BatchNorm statistics + running stats, FIN = 1: backward sums + dgamma/dbeta
constexpr int RG = 32, CL = 8;
template <int FIN>
__global__ void __cluster_dims__(1, CL, 1) __launch_bounds__(32 * RG)
bn_reduce_kernel(const float* __restrict__ partial, int nblk, int d, long count, float eps, float momentum, float* __restrict__ o0,
                 float* __restrict__ o1, float* __restrict__ r0, float* __restrict__ r1, int64_t* __restrict__ nbt) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    __shared__ double sh[2][RG][33];
    __shared__ double slice[2][32];
    const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5, c = blockIdx.x * 32 + cx, rank = blockIdx.y;
    double s = 0.0, q = 0.0;
    if (c < d) {
#pragma unroll 4
        for (int i = rank * RG + ry; i < nblk; i += RG * CL) {
            s += (double)partial[(long)i * 2 * d + c];
            q += (double)partial[(long)i * 2 * d + d + c];
        }
    }
    sh[0][ry][cx] = s; sh[1][ry][cx] = q;
    __syncthreads();
    if (ry == 0) {
#pragma unroll
        for (int j = 1; j < RG; ++j) { s += sh[0][j][cx]; q += sh[1][j][cx]; }
        slice[0][cx] = s; slice[1][cx] = q;
    }
    cluster.sync();
    if (rank == 0 && ry == 0 && c < d) {
        for (int r = 1; r < CL; ++r) {
            const double* remote = cluster.map_shared_rank(&slice[0][0], r);
            s += remote[cx];
            q += remote[32 + cx];
        }
        if (FIN == 0) {
            const double mu = s / (double)count;
            double var = q / (double)count - mu * mu;
            if (var < 0.0) var = 0.0;
            o0[c] = (float)mu;
            o1[c] = (float)(1.0 / sqrt(var + (double)eps));
            if (r0) {
                const double unb = count > 1 ? var * (double)count / (double)(count - 1) : var;
                r0[c] = (float)((1.0 - momentum) * (double)r0[c] + momentum * mu);
                r1[c] = (float)((1.0 - momentum) * (double)r1[c] + momentum * unb);
                if (c == 0 && nbt) *nbt += 1;
            }
        } else {
            o0[c] = (float)s;       // sums[0:d]  = sum du
            o0[d + c] = (float)q;   // sums[d:2d] = sum du * zhat
            r0[c] += (float)q;      // dgamma
            r1[c] += (float)s;      // dbeta
        }
    }
    cluster.sync();  // the slices stay mapped until rank 0 has read them
}

__global__ void __launch_bounds__(128) bn_eval_stats_kernel(const float* __restrict__ running_mean, const float* __restrict__ running_var,
                                                            float eps, float* __restrict__ mean, float* __restrict__ rstd, int d) {
    const int c = blockIdx.x * 128 + threadIdx.x;
    if (c >= d) return;
    mean[c] = running_mean[c];
    rstd[c] = rsqrtf(running_var[c] + eps);
}

// ---------------------------------------------------------------- bwd 1 (fast): one thread = 4 channels x (32 / groups) rows
template <typename TD>
__global__ void __launch_bounds__(256) bn_swish_bwd_stats_kernel(const TD* __restrict__ da, const float* __restrict__ z,
                                                                 const float* __restrict__ mean, const float* __restrict__ rstd,
                                                                 const float* __restrict__ gamma, const float* __restrict__ beta,
                                                                 float* __restrict__ partial, long rows, int d) {
    LASR_PDL_SYNC();
    __shared__ __align__(16) float4 red[2][256];
    const int vpr = d >> 2;                                 // float4 chunks per row
    const long r0 = (long)blockIdx.x * TCH, r1 = min(rows, r0 + TCH);
    float* part = partial + (long)blockIdx.x * 2 * d;
    for (int cb = 0; cb < vpr; cb += 256) {                 // d <= 1024: one pass
        const int per = min(vpr - cb, 256);                 // chunks handled in this pass (power of two for the supported d)
        const int groups = 256 / per;                       // row groups
        const int cv = cb + (threadIdx.x % per), grp = threadIdx.x / per;
        float4 s = make_float4(0, 0, 0, 0), q = make_float4(0, 0, 0, 0);
        if (grp < groups) {
            const int c = cv * 4;
            const float4 m = *reinterpret_cast<const float4*>(mean + c), rs = *reinterpret_cast<const float4*>(rstd + c);
            const float4 ga = *reinterpret_cast<const float4*>(gamma + c), be = *reinterpret_cast<const float4*>(beta + c);
#pragma unroll 4
            for (long r = r0 + grp; r < r1; r += groups) {
                const float4 zz = *reinterpret_cast<const float4*>(z + r * d + c);
                const float4 g = ld4c<TD>(da + r * d + c);
                const float zh0 = (zz.x - m.x) * rs.x, zh1 = (zz.y - m.y) * rs.y, zh2 = (zz.z - m.z) * rs.z, zh3 = (zz.w - m.w) * rs.w;
                const float du0 = g.x * dswishf_(ga.x * zh0 + be.x), du1 = g.y * dswishf_(ga.y * zh1 + be.y);
                const float du2 = g.z * dswishf_(ga.z * zh2 + be.z), du3 = g.w * dswishf_(ga.w * zh3 + be.w);
                s.x += du0; s.y += du1; s.z += du2; s.w += du3;
                q.x += du0 * zh0; q.y += du1 * zh1; q.z += du2 * zh2; q.w += du3 * zh3;
            }
        }
        red[0][threadIdx.x] = s; red[1][threadIdx.x] = q;
        __syncthreads();
        if (grp == 0) {
            for (int g2 = 1; g2 < groups; ++g2) {
                const float4 a = red[0][threadIdx.x + g2 * per], b2 = red[1][threadIdx.x + g2 * per];
                s.x += a.x; s.y += a.y; s.z += a.z; s.w += a.w;
                q.x += b2.x; q.y += b2.y; q.z += b2.z; q.w += b2.w;
            }
            *reinterpret_cast<float4*>(part + cv * 4) = s;
            *reinterpret_cast<float4*>(part + d + cv * 4) = q;
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------- bwd 2 (fast)
// Same tiling as the forward kernel (FT x FC, thread = one channel x FT/4 steps).  shared: dz tile [FWIN][FC], g tile [FWIN][FC],
// sigmoid(gate) tile [FT][FC]; the dz tile is reused as the reduction buffer.
struct BwdSmem {
    float dz[FWIN][FC];
    float g[FWIN][FC];
    float sg[FT][FC];
    float wt[FC * KW];
};

template <typename TD>
__global__ void __launch_bounds__(256, 3) dwconv_glu_bwd_kernel(const TD* __restrict__ da, const float* __restrict__ z,
                                                                const TD* __restrict__ y2, long ldy, const float* __restrict__ mean,
                                                                const float* __restrict__ rstd, const float* __restrict__ gamma,
                                                                const float* __restrict__ beta, const float* __restrict__ sums,
                                                                const float* __restrict__ w, TD* __restrict__ dy2, long lddy,
                                                                float* __restrict__ dw, float* __restrict__ dbias,
                                                                float* __restrict__ colsum, float* __restrict__ wpartial, int T, int d,
                                                                float inv_count) {
    LASR_PDL_SYNC();
    extern __shared__ __align__(16) uint8_t smem_raw[];
    BwdSmem& sm = *reinterpret_cast<BwdSmem*>(smem_raw);
    const int b = blockIdx.y, c0 = blockIdx.z * FC, t0 = blockIdx.x * FT;
    for (int i = threadIdx.x; i < FC * KW; i += 256) sm.wt[i] = (c0 + i / KW < d) ? w[(long)c0 * KW + i] : 0.f;
    // phase 1: dz (BatchNorm + Swish backward) and g (GLU output) for the halo window, sigmoid(gate) for the centre rows.
    // A thread keeps one channel quad for all its rows: the per-channel constants are loaded once.
    {
        const int cv = (threadIdx.x & 15) * 4, rbase = threadIdx.x >> 4, c = c0 + cv;
        const bool cok = c < d;
        float4 m = make_float4(0.f, 0.f, 0.f, 0.f), rs = m, ga = m, be = m, su = m, sq = m;
        if (cok) {
            m = *reinterpret_cast<const float4*>(mean + c); rs = *reinterpret_cast<const float4*>(rstd + c);
            ga = *reinterpret_cast<const float4*>(gamma + c); be = *reinterpret_cast<const float4*>(beta + c);
            su = *reinterpret_cast<const float4*>(sums + c); sq = *reinterpret_cast<const float4*>(sums + d + c);
            su.x *= inv_count; su.y *= inv_count; su.z *= inv_count; su.w *= inv_count;
            sq.x *= inv_count; sq.y *= inv_count; sq.z *= inv_count; sq.w *= inv_count;
        }
        constexpr int NIT = (FWIN + 15) / 16;
#pragma unroll
        for (int it = 0; it < NIT; ++it) {
            const int r = rbase + 16 * it, tt = t0 - HALO + r;
            if (r >= FWIN) break;
            float4 dzv = make_float4(0.f, 0.f, 0.f, 0.f), gv = dzv, sgv = dzv;
            if (tt >= 0 && tt < T && cok) {
                const long rr = (long)b * T + tt;
                const float4 zz = *reinterpret_cast<const float4*>(z + rr * d + c);
                const float4 gd = ld4c<TD>(da + rr * d + c);
                const TD* row = y2 + rr * ldy + c;
                const float4 v = ld4c<TD>(row), gate = ld4c<TD>(row + d);
                const float zh0 = (zz.x - m.x) * rs.x, zh1 = (zz.y - m.y) * rs.y, zh2 = (zz.z - m.z) * rs.z, zh3 = (zz.w - m.w) * rs.w;
                dzv.x = ga.x * rs.x * (gd.x * dswishf_(ga.x * zh0 + be.x) - su.x - zh0 * sq.x);
                dzv.y = ga.y * rs.y * (gd.y * dswishf_(ga.y * zh1 + be.y) - su.y - zh1 * sq.y);
                dzv.z = ga.z * rs.z * (gd.z * dswishf_(ga.z * zh2 + be.z) - su.z - zh2 * sq.z);
                dzv.w = ga.w * rs.w * (gd.w * dswishf_(ga.w * zh3 + be.w) - su.w - zh3 * sq.w);
                sgv = make_float4(sigmoidf_(gate.x), sigmoidf_(gate.y), sigmoidf_(gate.z), sigmoidf_(gate.w));
                gv = make_float4(v.x * sgv.x, v.y * sgv.y, v.z * sgv.z, v.w * sgv.w);
            }
            *reinterpret_cast<float4*>(&sm.dz[r][cv]) = dzv;
            *reinterpret_cast<float4*>(&sm.g[r][cv]) = gv;
            if (r >= HALO && r < HALO + FT) *reinterpret_cast<float4*>(&sm.sg[r - HALO][cv]) = sgv;
        }
    }
    __syncthreads();
    // phase 2
    const int c = threadIdx.x & (FC - 1), qtr = threadIdx.x >> 6, cg = c0 + c;
    const bool act = cg < d;
    float aw[KW];
#pragma unroll
    for (int k = 0; k < KW; ++k) aw[k] = 0.f;
    float ab = 0.f, csv = 0.f, csg = 0.f;
    if (act) {
        const int tb = qtr * FQ;
        {
            float wk[KW];
#pragma unroll
            for (int k = 0; k < KW; ++k) wk[k] = sm.wt[c * KW + k];
            float dzw[FQ + KW - 1];
#pragma unroll
            for (int j = 0; j < FQ + KW - 1; ++j) dzw[j] = sm.dz[tb + j][c];
            TD* orow = dy2 + ((long)b * T + t0 + tb) * lddy + cg;
#pragma unroll
            for (int i = 0; i < FQ; ++i) {
                // z[t'] = sum_k w[k] g[t'+k-7]  =>  dg[t] = sum_k w[k] dz[t+7-k]   (window index i + 14 - k)
                float dg = 0.f;
#pragma unroll
                for (int k = 0; k < KW; ++k) dg = fmaf(wk[k], dzw[i + KW - 1 - k], dg);
                if (t0 + tb + i < T) {
                    const float sg = sm.sg[tb + i][c], gg = sm.g[tb + i + HALO][c];
                    const float v0 = dg * sg;                  // d(value half)
                    const float g0 = dg * gg * (1.f - sg);     // d(gate half): v*s*(1-s) = g*(1-s)
                    orow[(long)i * lddy] = from_f32<TD>(v0);
                    orow[(long)i * lddy + d] = from_f32<TD>(g0);
                    csv += v0;
                    csg += g0;
                }
            }
        }
        {
            // dw[k] += dz[t] * g[t+k-7] ; db += dz[t]     (dz[t] = 0 beyond the utterance end)
            float gw[FQ + KW - 1];
#pragma unroll
            for (int j = 0; j < FQ + KW - 1; ++j) gw[j] = sm.g[tb + j][c];
#pragma unroll
            for (int i = 0; i < FQ; ++i) {
                const float dzc = sm.dz[tb + i + HALO][c];
#pragma unroll
                for (int k = 0; k < KW; ++k) aw[k] = fmaf(dzc, gw[i + k], aw[k]);
                ab += dzc;
            }
        }
    }
    __syncthreads();  // every thread is done with the tiles: reuse sm.dz as the reduction buffer [4][NRED][FC]
    float* red = &sm.dz[0][0];
    {
        float* mine = red + (long)qtr * NRED * FC;
#pragma unroll
        for (int k = 0; k < KW; ++k) mine[k * FC + c] = aw[k];
        mine[KW * FC + c] = ab;
        mine[(KW + 1) * FC + c] = csv;
        mine[(KW + 2) * FC + c] = csg;
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < NRED * FC; idx += 256) {
        const int k = idx / FC, cc = idx % FC;
        if (c0 + cc >= d) continue;
        const float v = (red[idx] + red[NRED * FC + idx]) + (red[2 * NRED * FC + idx] + red[3 * NRED * FC + idx]);
        if (wpartial) {  // deterministic two-stage reduction: [CTA (b, chunk)][NRED][d], summed by dwconv_reduce_kernel
            wpartial[(((long)b * gridDim.x + blockIdx.x) * NRED + k) * d + c0 + cc] = v;
            continue;
        }
        if (k < KW) atomicAdd(dw + (long)(c0 + cc) * KW + k, v);
        else if (k == KW) atomicAdd(dbias + c0 + cc, v);
        else if (colsum) atomicAdd(colsum + (k == KW + 1 ? 0 : d) + c0 + cc, v);
    }
}

// (A streaming variant of the backward kernel -- the scheme of glu_dwconv_fwd_stream_kernel with three more rings -- was built and
//  measured: 76 us against 63 us for the tiled kernel above at C2 / B = 126.  Both execute ~40 M warp instructions; the streaming one
//  needs 105 KB of shared memory and 119 registers, i.e. 2 CTAs per SM, and the kernel is bound by its instruction stream (issue
//  slots 56-63 % busy), not by loads in flight.  profiles/r2_convmod_stream.txt.)

// second stage of the depthwise-weight / bias / pointwise-bias gradient: block (32 channels, RG row groups), grid (d/32, KW+3)
// (already 144 CTAs of 1024 threads at d = 256: a cluster split like bn_reduce's measured 3x slower here)
__global__ void __launch_bounds__(32 * RG) dwconv_reduce_kernel(const float* __restrict__ wpartial, int nblk, int d, float* __restrict__ dw,
                                                                float* __restrict__ dbias, float* __restrict__ colsum) {
    LASR_PDL_SYNC();
    __shared__ float sh[RG][33];
    const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5, c = blockIdx.x * 32 + cx, k = blockIdx.y;
    float s = 0.f;
    if (c < d) {
#pragma unroll 4
        for (int i = ry; i < nblk; i += RG) s += wpartial[((long)i * NRED + k) * d + c];
    }
    sh[ry][cx] = s;
    __syncthreads();
    if (ry != 0 || c >= d) return;
#pragma unroll
    for (int j = 1; j < RG; ++j) s += sh[j][cx];
    if (k < KW) dw[(long)c * KW + k] += s;
    else if (k == KW) dbias[c] += s;
    else if (colsum) colsum[(k == KW + 1 ? 0 : d) + c] += s;
}

}  // namespace lasr

extern "C" {
using namespace lasr;

static inline bool fast_d(int d) { return d % 4 == 0; }
static inline bool pow2_rows(int d) { const int v = d / 4; return d % 4 == 0 && v >= 1 && v <= 256 && (v & (v - 1)) == 0; }

extern "C++" {
template <bool LENS>
static int glu_dwconv_fwd_launch(const void* y2, int dtype, int64_t ldy, const float* w, const float* bias, float* z, float* partial,
                                 int B, int T, int d, const int64_t* lens, void* stream) {
    LASR_REQUIRE(y2 && w && bias && z && partial && B > 0 && T > 0 && d > 0 && d % 2 == 0 && ldy % 2 == 0, "glu_dwconv_fwd: bad args");
    cudaStream_t st = (cudaStream_t)stream;
    const bool fast = fast_d(d) && ldy % 4 == 0 && ((uintptr_t)y2 & 15) == 0 && ((uintptr_t)z & 15) == 0;
    if (dtype == LASR_BF16 && d % SCH == 0 && ldy % 8 == 0 && ((uintptr_t)y2 & 15) == 0) {
        launch_pdl(glu_dwconv_fwd_stream_kernel<LENS>, dim3(d / SCH, B), 256, 0, st, (const bf16*)y2, ldy, w, bias, z, partial, T, d, lens);
        return check_launch("glu_dwconv_fwd");
    }
    if (fast) {
        dim3 grid(ceil_div(T, FT), B, ceil_div(d, FC));
        if (dtype == LASR_F32) launch_pdl(glu_dwconv_fwd_kernel<float, LENS>, grid, 256, 0, st, (const float*)y2, ldy, w, bias, z, partial, T, d, lens);
        else if (dtype == LASR_BF16) launch_pdl(glu_dwconv_fwd_kernel<bf16, LENS>, grid, 256, 0, st, (const bf16*)y2, ldy, w, bias, z, partial, T, d, lens);
        else { set_error("glu_dwconv_fwd: bad dtype"); return LASR_ERR_UNSUPPORTED; }
    } else {
        dim3 grid(ceil_div(T, TCH), B);
        if (dtype == LASR_F32) glu_dwconv_fwd_generic<float, LENS><<<grid, 128, 0, st>>>((const float*)y2, ldy, w, bias, z, partial, T, d, lens);
        else if (dtype == LASR_BF16) glu_dwconv_fwd_generic<bf16, LENS><<<grid, 128, 0, st>>>((const bf16*)y2, ldy, w, bias, z, partial, T, d, lens);
        else { set_error("glu_dwconv_fwd: bad dtype"); return LASR_ERR_UNSUPPORTED; }
    }
    return check_launch("glu_dwconv_fwd");
}
}  // extern "C++"

/* partial: B * ceil(T/32) * 2 * d floats */
int lasr_glu_dwconv_fwd(const void* y2, int dtype, int64_t ldy, const float* w, const float* bias, float* z, float* partial,
                        int B, int T, int d, void* stream) {
    return glu_dwconv_fwd_launch<false>(y2, dtype, ldy, w, bias, z, partial, B, T, d, nullptr, stream);
}

int lasr_glu_dwconv_fwd_lens(const void* y2, int dtype, int64_t ldy, const float* w, const float* bias, float* z, float* partial,
                             int B, int T, int d, const int64_t* lens, void* stream) {
    LASR_REQUIRE(lens, "glu_dwconv_fwd_lens: lens is required");
    return glu_dwconv_fwd_launch<true>(y2, dtype, ldy, w, bias, z, partial, B, T, d, lens, stream);
}

int lasr_bn_finalize(const float* partial, int nblk, int d, int64_t count, float eps, float momentum, float* mean, float* rstd,
                     float* running_mean, float* running_var, int64_t* num_batches_tracked, int training, void* stream) {
    LASR_REQUIRE(mean && rstd && d > 0 && (training ? (partial && nblk > 0 && count > 0) : (running_mean && running_var)), "bn_finalize: bad args");
    LASR_REQUIRE(!training || ((running_mean != nullptr) == (running_var != nullptr)), "bn_finalize: running stats come in pairs");
    cudaStream_t st = (cudaStream_t)stream;
    if (!training) bn_eval_stats_kernel<<<ceil_div(d, 128), 128, 0, st>>>(running_mean, running_var, eps, mean, rstd, d);
    else bn_reduce_kernel<0><<<dim3(ceil_div(d, 32), CL), 32 * RG, 0, st>>>(partial, nblk, d, count, eps, momentum, mean, rstd, running_mean, running_var,
                                                             num_batches_tracked);
    return check_launch("bn_finalize");
}

int lasr_bn_swish_fwd(const float* z, const float* mean, const float* rstd, const float* gamma, const float* beta, void* a,
                      int dtype, int64_t rows, int d, void* stream) {
    LASR_REQUIRE(z && mean && rstd && gamma && beta && a && rows > 0 && d % 2 == 0, "bn_swish_fwd: bad args");
    const long n = rows * d;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype != LASR_F32 && dtype != LASR_BF16) { set_error("bn_swish_fwd: bad dtype"); return LASR_ERR_UNSUPPORTED; }
    const bool vec = d % 4 == 0 && (((uintptr_t)z | (uintptr_t)mean | (uintptr_t)rstd | (uintptr_t)gamma | (uintptr_t)beta | (uintptr_t)a) & 15) == 0;
    if (vec) {
        const long threads = (long)(d >> 2) * ((rows + 3) / 4);
        if (dtype == LASR_F32) launch_pdl(bn_swish_fwd_vec_kernel<float>, ceil_div(threads, 256), 256, 0, st, z, mean, rstd, gamma, beta, (float*)a, rows, d);
        else launch_pdl(bn_swish_fwd_vec_kernel<bf16>, ceil_div(threads, 256), 256, 0, st, z, mean, rstd, gamma, beta, (bf16*)a, rows, d);
    } else if (dtype == LASR_F32) bn_swish_fwd_kernel<float><<<ceil_div(n / 2, 256), 256, 0, st>>>(z, mean, rstd, gamma, beta, (float*)a, n, d);
    else bn_swish_fwd_kernel<bf16><<<ceil_div(n / 2, 256), 256, 0, st>>>(z, mean, rstd, gamma, beta, (bf16*)a, n, d);
    return check_launch("bn_swish_fwd");
}

/* partial: ceil(rows/32) * 2 * d floats; sums: 2 * d floats */
int lasr_bn_swish_bwd_stats(const void* da, int dtype, const float* z, const float* mean, const float* rstd, const float* gamma,
                            const float* beta, float* partial, float* sums, float* dgamma, float* dbeta, int64_t rows, int d,
                            void* stream) {
    LASR_REQUIRE(da && z && mean && rstd && gamma && beta && partial && sums && dgamma && dbeta && rows > 0 && d % 2 == 0, "bn_swish_bwd_stats: bad args");
    const int nblk = ceil_div(rows, TCH);
    cudaStream_t st = (cudaStream_t)stream;
    const bool fast = pow2_rows(d) && ((uintptr_t)da & 15) == 0 && ((uintptr_t)z & 15) == 0 && ((uintptr_t)partial & 15) == 0 &&
                      (((uintptr_t)mean | (uintptr_t)rstd | (uintptr_t)gamma | (uintptr_t)beta) & 15) == 0;
    if (dtype != LASR_F32 && dtype != LASR_BF16) { set_error("bn_swish_bwd_stats: bad dtype"); return LASR_ERR_UNSUPPORTED; }
    if (fast) {
        if (dtype == LASR_F32) launch_pdl(bn_swish_bwd_stats_kernel<float>, nblk, 256, 0, st, (const float*)da, z, mean, rstd, gamma, beta, partial, rows, d);
        else launch_pdl(bn_swish_bwd_stats_kernel<bf16>, nblk, 256, 0, st, (const bf16*)da, z, mean, rstd, gamma, beta, partial, rows, d);
    } else {
        if (dtype == LASR_F32) bn_swish_bwd_stats_generic<float><<<nblk, 128, 0, st>>>((const float*)da, z, mean, rstd, gamma, beta, partial, rows, d);
        else bn_swish_bwd_stats_generic<bf16><<<nblk, 128, 0, st>>>((const bf16*)da, z, mean, rstd, gamma, beta, partial, rows, d);
    }
    int rc = check_launch("bn_swish_bwd_stats");
    if (rc) return rc;
    bn_reduce_kernel<1><<<dim3(ceil_div(d, 32), CL), 32 * RG, 0, st>>>(partial, nblk, d, 0, 0.f, 0.f, sums, nullptr, dgamma, dbeta, nullptr);
    return check_launch("bn_bwd_finalize");
}

int lasr_dwconv_glu_bwd(const void* da, const float* z, const void* y2, int dtype, int64_t ldy, const float* mean, const float* rstd,
                        const float* gamma, const float* beta, const float* sums, const float* w, void* dy2, int64_t lddy, float* dw,
                        float* dbias, float* colsum, float* wpartial, int B, int T, int d, void* stream) {
    LASR_REQUIRE(da && z && y2 && mean && rstd && gamma && beta && sums && w && dy2 && dw && dbias && B > 0 && T > 0 && d % 2 == 0 &&
                     ldy % 2 == 0 && lddy % 2 == 0, "dwconv_glu_bwd: bad args");
    const float inv = 1.f / (float)((long)B * T);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype != LASR_F32 && dtype != LASR_BF16) { set_error("dwconv_glu_bwd: bad dtype"); return LASR_ERR_UNSUPPORTED; }
    const bool fast = fast_d(d) && ldy % 4 == 0 && lddy % 2 == 0 &&
                      (((uintptr_t)da | (uintptr_t)z | (uintptr_t)y2 | (uintptr_t)mean | (uintptr_t)rstd | (uintptr_t)gamma | (uintptr_t)beta |
                        (uintptr_t)sums) & 15) == 0;
    if (fast) {
        dim3 grid(ceil_div(T, FT), B, ceil_div(d, FC));
        const int smem = (int)sizeof(BwdSmem);
        static bool configured = false;
        if (!configured) {
            if (cudaFuncSetAttribute(dwconv_glu_bwd_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess ||
                cudaFuncSetAttribute(dwconv_glu_bwd_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess)
                return check_launch("dwconv_glu_bwd smem attr");
            configured = true;
        }
        if (dtype == LASR_F32)
            launch_pdl(dwconv_glu_bwd_kernel<float>, grid, 256, smem, st, (const float*)da, z, (const float*)y2, ldy, mean, rstd, gamma, beta, sums, w,
                                                                 (float*)dy2, lddy, dw, dbias, colsum, wpartial, T, d, inv);
        else
            launch_pdl(dwconv_glu_bwd_kernel<bf16>, grid, 256, smem, st, (const bf16*)da, z, (const bf16*)y2, ldy, mean, rstd, gamma, beta, sums, w,
                                                                (bf16*)dy2, lddy, dw, dbias, colsum, wpartial, T, d, inv);
        int rc = check_launch("dwconv_glu_bwd");
        if (rc || !wpartial) return rc;
        launch_pdl(dwconv_reduce_kernel, dim3(ceil_div(d, 32), KW + 3), 32 * RG, 0, st, wpartial, B * ceil_div(T, FT), d, dw, dbias, colsum);
        return check_launch("dwconv_reduce");
    }
    dim3 grid(ceil_div(T, TCH), B);
    if (dtype == LASR_F32)
        dwconv_glu_bwd_generic<float><<<grid, 128, 0, st>>>((const float*)da, z, (const float*)y2, ldy, mean, rstd, gamma, beta, sums, w,
                                                           (float*)dy2, lddy, dw, dbias, T, d, inv);
    else
        dwconv_glu_bwd_generic<bf16><<<grid, 128, 0, st>>>((const bf16*)da, z, (const bf16*)y2, ldy, mean, rstd, gamma, beta, sums, w,
                                                          (bf16*)dy2, lddy, dw, dbias, T, d, inv);
    int rc = check_launch("dwconv_glu_bwd");
    if (rc || !colsum) return rc;
    return lasr_act_bwd(dy2, lddy, nullptr, 0, nullptr, 0, colsum, B * T, 2 * d, LASR_ACT_NONE, 1.f, dtype, stream);
}

}  // extern "C"
