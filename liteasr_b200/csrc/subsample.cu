// Conv2d subsampling (nets/subsampling.py:32-35,42-46) in channel-last layout.
//   conv1: Conv2d(1 -> d, 3x3, stride 2) + ReLU, direct (K = 9, HBM-bound):  (B,T,F) -> (B,T1,F1,d)
//   conv2: Conv2d(d -> d, 3x3, stride 2) + ReLU = GEMM over an im2col matrix (B*T2*F2, 9d) whose K index is
//          (kh, kw, c_in); with channel-last activations every (kh, kw) patch is d contiguous elements, so
//          im2col / col2im are pure 128-bit copy kernels and the GEMM output (B,T2,F2*d) is already the
//          (B,T',F2*d) matrix the output Linear consumes (its weight columns are permuted once per step).
//   backward: col2im gather fused with conv1's ReLU mask; conv1 weight/bias gradient by direct accumulation.
#include "common.cuh"

namespace lasr {

// ---------------------------------------------------------------- conv1 forward
template <typename TD>
__global__ void __launch_bounds__(256) conv1_fwd_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                        const float* __restrict__ bias, TD* __restrict__ h1, int T, int F,
                                                        int T1, int F1, int d) {
    extern __shared__ float xs[];  // 3 rows x F
    const int b = blockIdx.y, t1 = blockIdx.x;
    for (int i = threadIdx.x; i < 3 * F; i += blockDim.x) xs[i] = x[((long)b * T + 2 * t1) * F + i];
    __syncthreads();
    for (int c = threadIdx.x; c < d; c += blockDim.x) {
        float wk[9];
#pragma unroll
        for (int k = 0; k < 9; ++k) wk[k] = w[c * 9 + k];
        const float bc = bias[c];
        TD* out = h1 + (((long)b * T1 + t1) * F1) * d + c;
        for (int f = 0; f < F1; ++f) {
            float a = bc;
#pragma unroll
            for (int kh = 0; kh < 3; ++kh)
#pragma unroll
                for (int kw = 0; kw < 3; ++kw) a = fmaf(wk[kh * 3 + kw], xs[kh * F + 2 * f + kw], a);
            out[(long)f * d] = from_f32<TD>(fmaxf(a, 0.f));
        }
    }
}

// ---------------------------------------------------------------- conv1 backward (weights only; the input is data)
template <typename TD>
__global__ void __launch_bounds__(256) conv1_bwd_kernel(const float* __restrict__ x, const TD* __restrict__ dh1,
                                                        float* __restrict__ dw, float* __restrict__ dbias, int T, int F, int T1,
                                                        int F1, int d, int rows_per_cta, long total_rows) {
    extern __shared__ float xs[];  // 3 rows x F
    const long r0 = (long)blockIdx.x * rows_per_cta, r1 = min(total_rows, r0 + rows_per_cta);
    // each thread owns channels c, c + blockDim, ... (at most 4 supported: d <= 1024)
    float acc[4][10];
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int k = 0; k < 10; ++k) acc[j][k] = 0.f;
    for (long r = r0; r < r1; ++r) {
        const int b = (int)(r / T1), t1 = (int)(r % T1);
        __syncthreads();
        for (int i = threadIdx.x; i < 3 * F; i += blockDim.x) xs[i] = x[((long)b * T + 2 * t1) * F + i];
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int c = threadIdx.x + j * blockDim.x;
            if (c < d) {
                const TD* g = dh1 + (r * F1) * d + c;
                for (int f = 0; f < F1; ++f) {
                    const float gv = to_f32<TD>(g[(long)f * d]);
#pragma unroll
                    for (int kh = 0; kh < 3; ++kh)
#pragma unroll
                        for (int kw = 0; kw < 3; ++kw) acc[j][kh * 3 + kw] = fmaf(gv, xs[kh * F + 2 * f + kw], acc[j][kh * 3 + kw]);
                    acc[j][9] += gv;
                }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int c = threadIdx.x + j * blockDim.x;
        if (c < d) {
#pragma unroll
            for (int k = 0; k < 9; ++k) atomicAdd(dw + c * 9 + k, acc[j][k]);
            atomicAdd(dbias + c, acc[j][9]);
        }
    }
}

// ---------------------------------------------------------------- im2col (stride 2, 3x3), 16-byte vectors
template <typename TD>
__global__ void __launch_bounds__(256) im2col_kernel(const TD* __restrict__ h1, TD* __restrict__ col, int B, int T1, int F1,
                                                     int T2, int F2, int d) {
    constexpr int VEC = 16 / sizeof(TD);
    const int vpp = d / VEC;  // vectors per patch
    const long total = (long)B * T2 * F2 * 9 * vpp;
    for (long i = (long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long)gridDim.x * 256) {
        long r = i;
        const int v = (int)(r % vpp); r /= vpp;
        const int kk = (int)(r % 9); r /= 9;
        const int f2 = (int)(r % F2); r /= F2;
        const int t2 = (int)(r % T2); r /= T2;
        const int b = (int)r;
        const int kh = kk / 3, kw = kk % 3;
        const uint4 val = *reinterpret_cast<const uint4*>(h1 + ((((long)b * T1 + 2 * t2 + kh) * F1 + 2 * f2 + kw) * d) + v * VEC);
        *reinterpret_cast<uint4*>(col + i * VEC) = val;
    }
}

// ---------------------------------------------------------------- col2im gather + ReLU mask of conv1's output
template <typename TD>
__global__ void __launch_bounds__(256) col2im_relu_kernel(const TD* __restrict__ dcol, const TD* __restrict__ h1,
                                                          TD* __restrict__ dh1, int B, int T1, int F1, int T2, int F2, int d) {
    const int vpp = d / 4;
    const long total = (long)B * T1 * F1 * vpp;
    for (long i = (long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long)gridDim.x * 256) {
        long r = i;
        const int v = (int)(r % vpp); r /= vpp;
        const int f1 = (int)(r % F1); r /= F1;
        const int t1 = (int)(r % T1); r /= T1;
        const int b = (int)r;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
        for (int kh = 0; kh < 3; ++kh) {
            const int tn = t1 - kh;
            if (tn < 0 || (tn & 1) || (tn >> 1) >= T2) continue;
#pragma unroll
            for (int kw = 0; kw < 3; ++kw) {
                const int fn = f1 - kw;
                if (fn < 0 || (fn & 1) || (fn >> 1) >= F2) continue;
                const long row = ((long)b * T2 + (tn >> 1)) * F2 + (fn >> 1);
                const TD* p = dcol + row * 9 * d + (kh * 3 + kw) * d + v * 4;
                if constexpr (sizeof(TD) == 4) {
                    const float4 q = *reinterpret_cast<const float4*>(p);
                    a0 += q.x; a1 += q.y; a2 += q.z; a3 += q.w;
                } else {
                    const uint2 u = *reinterpret_cast<const uint2*>(p);
                    const __nv_bfloat162 lo = *reinterpret_cast<const __nv_bfloat162*>(&u.x), hi = *reinterpret_cast<const __nv_bfloat162*>(&u.y);
                    a0 += __low2float(lo); a1 += __high2float(lo); a2 += __low2float(hi); a3 += __high2float(hi);
                }
            }
        }
        const long off = i * 4;
        const float m0 = to_f32<TD>(h1[off]) > 0.f, m1 = to_f32<TD>(h1[off + 1]) > 0.f;
        const float m2 = to_f32<TD>(h1[off + 2]) > 0.f, m3 = to_f32<TD>(h1[off + 3]) > 0.f;
        dh1[off] = from_f32<TD>(a0 * m0); dh1[off + 1] = from_f32<TD>(a1 * m1);
        dh1[off + 2] = from_f32<TD>(a2 * m2); dh1[off + 3] = from_f32<TD>(a3 * m3);
    }
}


// =================================================================================================
// parity-plane variants (feed the implicit-GEMM conv2, gemm_tc.cu::conv2_tc_dispatch)
//   h1p[b][pt*2+pf][u*V + v][c]  with t1 = 2u+pt, f1 = 2v+pf, U = ceil(T1/2), V = ceil(F1/2); slots without a (t1,f1) are ZERO.
// =================================================================================================
// CTA = PR_ROWS consecutive t1 rows of one utterance (t1 in [0, 2U)); the 2*PR_ROWS+1 input rows and the transposed conv1
// weights are staged in shared memory once; thread = 4 channels x every ng-th (row, frequency slot) task; 8-byte stores.
constexpr int PR_ROWS = 8;
template <int DUMMY>
__global__ void __launch_bounds__(256) conv1_fwd_planes_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                               const float* __restrict__ bias, bf16* __restrict__ h1p, int T, int F,
                                                               int T1, int F1, int U, int V, int d) {
    extern __shared__ __align__(16) float smf[];
    float* ws = smf;                  // [9][d] (tap-major: a thread reads its 4 channels as one float4)
    float* xs = smf + 9 * d;          // (2 * PR_ROWS + 1) rows x F
    const int b = blockIdx.y, t10 = blockIdx.x * PR_ROWS;
    const int quads = d >> 2, q = threadIdx.x % quads, g = threadIdx.x / quads, ng = 256 / quads;
    const long plane_rows = (long)U * V;
    for (int i = threadIdx.x; i < 9 * d; i += 256) ws[(i % 9) * d + i / 9] = w[i];
    const int xrows = 2 * PR_ROWS + 1;
    for (int i = threadIdx.x; i < xrows * F; i += 256) {
        const int tr = 2 * t10 + i / F;
        xs[i] = tr < T ? x[((long)b * T + tr) * F + i % F] : 0.f;
    }
    __syncthreads();
    float4 wk[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) wk[k] = *reinterpret_cast<const float4*>(ws + k * d + 4 * q);
    const float4 bc = *reinterpret_cast<const float4*>(bias + 4 * q);
    bf16* hb = h1p + (long)b * 4 * plane_rows * d + 4 * q;
    for (int i = 0; i < PR_ROWS; ++i) {
        const int t1 = t10 + i;
        if (t1 >= 2 * U) break;
        const bool row_ok = t1 < T1;
        bf16* rowp = hb + ((long)((t1 & 1) * 2) * plane_rows + (long)(t1 >> 1) * V) * d;  // plane (pt, pf = 0), row u
        const float* xrow = xs + (2 * i) * F;
        for (int f = g; f < 2 * V; f += ng) {  // f1 slots 0 .. 2V-1 (the last one may not exist)
            uint2 o = make_uint2(0u, 0u);
            if (row_ok && f < F1) {
                float4 a = bc;
                const float* xr = xrow + 2 * f;
#pragma unroll
                for (int kh = 0; kh < 3; ++kh)
#pragma unroll
                    for (int kw = 0; kw < 3; ++kw) {
                        const float xv = xr[kh * F + kw];
                        const float4 ww = wk[kh * 3 + kw];
                        a.x = fmaf(ww.x, xv, a.x); a.y = fmaf(ww.y, xv, a.y); a.z = fmaf(ww.z, xv, a.z); a.w = fmaf(ww.w, xv, a.w);
                    }
                const __nv_bfloat162 lo = __floats2bfloat162_rn(fmaxf(a.x, 0.f), fmaxf(a.y, 0.f));
                const __nv_bfloat162 hi = __floats2bfloat162_rn(fmaxf(a.z, 0.f), fmaxf(a.w, 0.f));
                o.x = *reinterpret_cast<const uint32_t*>(&lo);
                o.y = *reinterpret_cast<const uint32_t*>(&hi);
            }
            *reinterpret_cast<uint2*>(rowp + ((long)(f & 1) * plane_rows + (f >> 1)) * d) = o;
        }
    }
}

// conv1 weight / bias gradient from dh1p (already ReLU-masked).  Persistent CTAs walk chunks of PR_ROWS t1 rows of one
// utterance; thread = 4 channels x every ng-th (row, frequency) task with the loads of 4 tasks in flight; 40 accumulators;
// CTA-level reduction through shared memory, then one atomic per value.
template <int DUMMY>
__global__ void __launch_bounds__(256, 3) conv1_bwd_planes_kernel(const float* __restrict__ x, const bf16* __restrict__ dh1p,
                                                               float* __restrict__ dw, float* __restrict__ dbias, int T, int F,
                                                               int T1, int F1, int U, int V, int d, int chunks_per_utt, long total_chunks) {
    extern __shared__ __align__(16) float sm[];  // (2 * PR_ROWS + 1) x F staging, reused as the reduction buffer
    const int quads = d >> 2, q = threadIdx.x % quads, g = threadIdx.x / quads, ng = 256 / quads;
    const long plane_rows = (long)U * V;
    float acc[4][10];
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int k = 0; k < 10; ++k) acc[j][k] = 0.f;
    const int xrows = 2 * PR_ROWS + 1;
    for (long ch = blockIdx.x; ch < total_chunks; ch += gridDim.x) {
        const int b = (int)(ch / chunks_per_utt), t10 = (int)(ch % chunks_per_utt) * PR_ROWS;
        __syncthreads();  // the previous chunk's readers are done with the staging buffer
        for (int i = threadIdx.x; i < xrows * F; i += 256) {
            const int tr = 2 * t10 + i / F;
            sm[i] = tr < T ? x[((long)b * T + tr) * F + i % F] : 0.f;
        }
        __syncthreads();
        const int nrow = min(PR_ROWS, T1 - t10);
        const bf16* hb = dh1p + (long)b * 4 * plane_rows * d + 4 * q;
        for (int i = 0; i < nrow; ++i) {
            const int t1 = t10 + i;
            const bf16* rowp = hb + ((long)((t1 & 1) * 2) * plane_rows + (long)(t1 >> 1) * V) * d;
            const float* xrow = sm + (2 * i) * F;
            for (int f0 = g; f0 < F1; f0 += 2 * ng) {  // two positions per trip: both loads are issued before the math
                const int f1b = f0 + ng;
                const bool two = f1b < F1;
                const uint2 raw0 = *reinterpret_cast<const uint2*>(rowp + ((long)(f0 & 1) * plane_rows + (f0 >> 1)) * d);
                uint2 raw1 = make_uint2(0u, 0u);
                if (two) raw1 = *reinterpret_cast<const uint2*>(rowp + ((long)(f1b & 1) * plane_rows + (f1b >> 1)) * d);
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const uint2 raw = e ? raw1 : raw0;
                    const __nv_bfloat162 lo = *reinterpret_cast<const __nv_bfloat162*>(&raw.x), hi = *reinterpret_cast<const __nv_bfloat162*>(&raw.y);
                    const float gv[4] = {__low2float(lo), __high2float(lo), __low2float(hi), __high2float(hi)};
                    const float* xr = xrow + 2 * (e ? (two ? f1b : f0) : f0);
#pragma unroll
                    for (int kh = 0; kh < 3; ++kh)
#pragma unroll
                        for (int kw = 0; kw < 3; ++kw) {
                            const float xv = xr[kh * F + kw];
#pragma unroll
                            for (int j = 0; j < 4; ++j) acc[j][kh * 3 + kw] = fmaf(gv[j], xv, acc[j][kh * 3 + kw]);
                        }
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[j][9] += gv[j];
                }
            }
        }
    }
    __syncthreads();
    // reduce the ng task groups through shared memory: red[g][c][10]
    float* red = sm;
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int k = 0; k < 10; ++k) red[((long)g * d + 4 * q + j) * 10 + k] = acc[j][k];
    __syncthreads();
    for (int i = threadIdx.x; i < d * 10; i += 256) {
        float s2 = 0.f;
        for (int gg = 0; gg < ng; ++gg) s2 += red[(long)gg * d * 10 + i];
        const int c = i / 10, k = i % 10;
        if (k < 9) atomicAdd(dw + c * 9 + k, s2);
        else atomicAdd(dbias + c, s2);
    }
}

int conv2_wgrad2_dispatch(const void* h1p, const void* dy, float* out, int B, int U, int V, int T2, int d, cudaStream_t st);
int conv2_tc_dispatch(int mode, int plane_class, const void* h1p, const void* w2, const float* bias, const void* dy, void* out,
                      int B, int U, int V, int T2, int d, int split_k, cudaStream_t st);
int conv1_wgrad_tc_dispatch(const float* x, const void* dh1p, float* dw, float* dbias, int B, int T, int F, int d, cudaStream_t st);
int conv1_fwd_tc_dispatch(const float* x, const float* w, const float* bias, void* h1p, int B, int T, int F, int d, cudaStream_t st);

}  // namespace lasr

extern "C" {
using namespace lasr;

int lasr_conv1_fwd(const float* x, const float* w, const float* bias, void* h1, int dtype, int B, int T, int F, int d, void* stream) {
    LASR_REQUIRE(x && w && bias && h1 && B > 0 && T >= 3 && F >= 3 && d > 0, "conv1_fwd: bad args");
    const int T1 = (T - 3) / 2 + 1, F1 = (F - 3) / 2 + 1;
    dim3 grid(T1, B);
    const size_t smem = 3 * F * sizeof(float);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == LASR_F32) conv1_fwd_kernel<float><<<grid, 256, smem, st>>>(x, w, bias, (float*)h1, T, F, T1, F1, d);
    else if (dtype == LASR_BF16) conv1_fwd_kernel<bf16><<<grid, 256, smem, st>>>(x, w, bias, (bf16*)h1, T, F, T1, F1, d);
    else { set_error("conv1_fwd: bad dtype"); return LASR_ERR_UNSUPPORTED; }
    return check_launch("conv1_fwd");
}

int lasr_conv1_bwd(const float* x, const void* dh1, int dtype, float* dw, float* dbias, int B, int T, int F, int d, void* stream) {
    LASR_REQUIRE(x && dh1 && dw && dbias && B > 0 && T >= 3 && F >= 3 && d > 0 && d <= 1024, "conv1_bwd: bad args");
    const int T1 = (T - 3) / 2 + 1, F1 = (F - 3) / 2 + 1;
    const long rows = (long)B * T1;
    const int rpc = 16;
    const size_t smem = 3 * F * sizeof(float);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == LASR_F32) conv1_bwd_kernel<float><<<ceil_div(rows, rpc), 256, smem, st>>>(x, (const float*)dh1, dw, dbias, T, F, T1, F1, d, rpc, rows);
    else if (dtype == LASR_BF16) conv1_bwd_kernel<bf16><<<ceil_div(rows, rpc), 256, smem, st>>>(x, (const bf16*)dh1, dw, dbias, T, F, T1, F1, d, rpc, rows);
    else { set_error("conv1_bwd: bad dtype"); return LASR_ERR_UNSUPPORTED; }
    return check_launch("conv1_bwd");
}

int lasr_im2col_s2(const void* h1, void* col, int dtype, int B, int T1, int F1, int d, void* stream) {
    LASR_REQUIRE(h1 && col && B > 0 && T1 >= 3 && F1 >= 3 && d % 8 == 0, "im2col: bad args (d%%8==0)");
    const int T2 = (T1 - 3) / 2 + 1, F2 = (F1 - 3) / 2 + 1;
    const long total = (long)B * T2 * F2 * 9 * (dtype == LASR_F32 ? d / 4 : d / 8);
    int grid = ceil_div(total, 256);
    if (grid > 148 * 32) grid = 148 * 32;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == LASR_F32) im2col_kernel<float><<<grid, 256, 0, st>>>((const float*)h1, (float*)col, B, T1, F1, T2, F2, d);
    else if (dtype == LASR_BF16) im2col_kernel<bf16><<<grid, 256, 0, st>>>((const bf16*)h1, (bf16*)col, B, T1, F1, T2, F2, d);
    else { set_error("im2col: bad dtype"); return LASR_ERR_UNSUPPORTED; }
    return check_launch("im2col");
}

int lasr_col2im_s2_relu(const void* dcol, const void* h1, void* dh1, int dtype, int B, int T1, int F1, int d, void* stream) {
    LASR_REQUIRE(dcol && h1 && dh1 && B > 0 && T1 >= 3 && F1 >= 3 && d % 4 == 0, "col2im: bad args");
    const int T2 = (T1 - 3) / 2 + 1, F2 = (F1 - 3) / 2 + 1;
    const long total = (long)B * T1 * F1 * (d / 4);
    int grid = ceil_div(total, 256);
    if (grid > 148 * 32) grid = 148 * 32;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == LASR_F32) col2im_relu_kernel<float><<<grid, 256, 0, st>>>((const float*)dcol, (const float*)h1, (float*)dh1, B, T1, F1, T2, F2, d);
    else if (dtype == LASR_BF16) col2im_relu_kernel<bf16><<<grid, 256, 0, st>>>((const bf16*)dcol, (const bf16*)h1, (bf16*)dh1, B, T1, F1, T2, F2, d);
    else { set_error("col2im: bad dtype"); return LASR_ERR_UNSUPPORTED; }
    return check_launch("col2im");
}

static inline bool planes_ok(int d) { return d % 64 == 0 && d >= 64 && d <= 1024 && 256 % (d / 4) == 0; }

int lasr_conv1_fwd_planes(const float* x, const float* w, const float* bias, void* h1p, int B, int T, int F, int d, void* stream) {
    LASR_REQUIRE(x && w && bias && h1p && B > 0 && T >= 7 && F >= 7 && planes_ok(d), "conv1_fwd_planes: bad args (d in {64,128,256,512,1024})");
    {
        // tensor-core path (csrc/conv1_fwd_tc.cu) for d = 128 / 256; LASR_CONV1_TC=0 keeps the SIMT kernel below
        const char* e = getenv("LASR_CONV1_TC");
        if (!(e && atoi(e) == 0)) {
            const int rc = conv1_fwd_tc_dispatch(x, w, bias, h1p, B, T, F, d, (cudaStream_t)stream);
            if (rc != LASR_ERR_UNSUPPORTED) return rc;
        }
    }
    const int T1 = (T - 3) / 2 + 1, F1 = (F - 3) / 2 + 1, U = (T1 + 1) / 2, V = (F1 + 1) / 2;
    dim3 grid(ceil_div(2 * U, PR_ROWS), B);
    const size_t smem = (9 * (size_t)d + (2 * PR_ROWS + 1) * (size_t)F) * sizeof(float);
    LASR_REQUIRE(smem <= 48 * 1024, "conv1_fwd_planes: F too large");
    conv1_fwd_planes_kernel<0><<<grid, 256, smem, (cudaStream_t)stream>>>(x, w, bias, (bf16*)h1p, T, F, T1, F1, U, V, d);
    return check_launch("conv1_fwd_planes");
}

int lasr_conv1_bwd_planes(const float* x, const void* dh1p, float* dw, float* dbias, int B, int T, int F, int d, void* stream) {
    LASR_REQUIRE(x && dh1p && dw && dbias && B > 0 && T >= 7 && F >= 7 && planes_ok(d), "conv1_bwd_planes: bad args");
    {
        // tensor-core path (csrc/conv1_wgrad_tc.cu) for d = 128 / 256 / 384 / 512; LASR_CONV1_TC=0 keeps the SIMT kernel below
        const char* e = getenv("LASR_CONV1_TC");
        if (!(e && atoi(e) == 0)) {
            const int rc = conv1_wgrad_tc_dispatch(x, dh1p, dw, dbias, B, T, F, d, (cudaStream_t)stream);
            if (rc != LASR_ERR_UNSUPPORTED) return rc;
        }
    }
    const int T1 = (T - 3) / 2 + 1, F1 = (F - 3) / 2 + 1, U = (T1 + 1) / 2, V = (F1 + 1) / 2;
    const int cpu = ceil_div(T1, PR_ROWS);
    const long chunks = (long)B * cpu;
    const int ng = 256 / (d / 4);
    size_t smem = (size_t)ng * d * 10 * sizeof(float);
    const size_t stage = (2 * PR_ROWS + 1) * (size_t)F * sizeof(float);
    if (smem < stage) smem = stage;
    static bool configured = false;
    if (!configured) {
        if (cudaFuncSetAttribute(conv1_bwd_planes_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024) != cudaSuccess)
            return check_launch("conv1_bwd_planes smem attr");
        configured = true;
    }
    LASR_REQUIRE(smem <= 100 * 1024, "conv1_bwd_planes: F too large");
    long grid = chunks < 148 * 3 ? chunks : 148 * 3;
    conv1_bwd_planes_kernel<0><<<(unsigned)grid, 256, smem, (cudaStream_t)stream>>>(x, (const bf16*)dh1p, dw, dbias, T, F, T1, F1, U, V, d, cpu,
                                                                                  chunks);
    return check_launch("conv1_bwd_planes");
}

/* Implicit-GEMM conv2 on the parity planes (bf16 / tcgen05 only).  Shapes: T1=(T-3)/2+1, F1=(F-3)/2+1, U=ceil(T1/2), V=ceil(F1/2),
 * T2=(T1-3)/2+1, F2=(F1-3)/2+1 = V-1.  w2k = conv.2.weight permuted to (co, kh, kw, ci) bf16. */
int lasr_conv2_fwd(const void* h1p, const void* w2k, const float* bias, void* h2p, int B, int T, int F, int d, void* stream) {
    LASR_REQUIRE(h1p && w2k && bias && h2p && planes_ok(d), "conv2_fwd: bad args");
    const int T1 = (T - 3) / 2 + 1, F1 = (F - 3) / 2 + 1, U = (T1 + 1) / 2, V = (F1 + 1) / 2, T2 = (T1 - 3) / 2 + 1;
    return conv2_tc_dispatch(1, 0, h1p, w2k, bias, nullptr, h2p, B, U, V, T2, d, 1, (cudaStream_t)stream);
}

int lasr_conv2_dgrad(const void* dy2p, const void* w2k, const void* h1p, void* dh1p, int B, int T, int F, int d, void* stream) {
    LASR_REQUIRE(dy2p && w2k && h1p && dh1p && planes_ok(d), "conv2_dgrad: bad args");
    const int T1 = (T - 3) / 2 + 1, F1 = (F - 3) / 2 + 1, U = (T1 + 1) / 2, V = (F1 + 1) / 2, T2 = (T1 - 3) / 2 + 1;
    for (int pl = 0; pl < 4; ++pl) {
        const int rc = conv2_tc_dispatch(2, pl, h1p, w2k, nullptr, dy2p, dh1p, B, U, V, T2, d, 1, (cudaStream_t)stream);
        if (rc) return rc;
    }
    return LASR_OK;
}

int lasr_conv2_wgrad(const void* dy2p, const void* h1p, float* dw2k, int B, int T, int F, int d, void* stream) {
    LASR_REQUIRE(dy2p && h1p && dw2k && planes_ok(d), "conv2_wgrad: bad args");
    const int T1 = (T - 3) / 2 + 1, F1 = (F - 3) / 2 + 1, U = (T1 + 1) / 2, V = (F1 + 1) / 2, T2 = (T1 - 3) / 2 + 1;
    if (d % 256 == 0) return conv2_wgrad2_dispatch(h1p, dy2p, dw2k, B, U, V, T2, d, (cudaStream_t)stream);  // CTA pairs (gemm2_wgrad.cu)
    return conv2_tc_dispatch(3, 0, h1p, nullptr, nullptr, dy2p, dw2k, B, U, V, T2, d, 1, (cudaStream_t)stream);
}

}  // extern "C"
