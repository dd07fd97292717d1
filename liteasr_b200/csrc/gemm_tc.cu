// bf16 GEMM on the 5th-gen tensor cores: tcgen05.mma with TMEM accumulators, TMA-fed smem ring.
//
//   C[b1,b2] (M,N) = alpha * act(A . B^T + bias) (+ res)        (or C += alpha * A.B^T with red.add)
//
// Persistent kernel: one CTA per SM walks the list of (batch, split, m-block, n-block) work units.
//   warp 0      TMA producer   : K streamed in 64-wide slabs through a STAGES-deep smem ring (runs ahead
//                                across work units, so short-K problems are not TMA-latency bound)
//   warp 1      MMA issuer     : tcgen05.mma 128 x BN x 16, fp32 accumulators in TMEM, two accumulator
//                                buffers (2 x 256 columns) so the epilogue of unit i overlaps the MMAs of i+1
//   warps 2..9  epilogue       : tcgen05.ld (thread = accumulator row) -> XOR-swizzled shared-memory transpose ->
//                                column phase (8 lanes per 128 B row segment): + bias (registers), optional
//                                pre-activation copy (aux), activation, alpha, + residual (coalesced, prefetched)
//                                -> row-contiguous vector stores; accumulate mode uses red.global.add.v4.f32
// BN is a run-time value (multiple of 16 up to 256; multiple of 64 when B is MN-major): it only changes the
// TMA box, the instruction descriptor and the ring stride, so N = 299 runs as 2 x 160 instead of 3 x 128.
// Both operands may be K-major (row-major (rows,K)) or MN-major (row-major (K,rows)); the difference is only
// in the TMA box shape, the UMMA shared-memory descriptor (LBO/SBO) and the instruction-descriptor major
// bits, so backward GEMMs (dgrad: B MN-major, wgrad: A and B MN-major) need no transposed copies.
#include <cuda.h>
#include <cudaTypedefs.h>

#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "common.cuh"
#include "philox.cuh"
#include "tc_ptx.cuh"

namespace lasr {

constexpr int BM = 128;
constexpr int BK = 64;  // 64 bf16 = 128 B = one SWIZZLE_128B row
constexpr int EPI_WARPS = 16;  // 4 per TMEM lane quarter (and per SM sub-partition): the epilogue is a latency chain per warp
constexpr int GEMM_THREADS = 64 + 32 * EPI_WARPS;
constexpr int UMMA_K = 16;
constexpr int A_BYTES = BM * BK * 2;
constexpr int MAX_STAGES = 8;
constexpr int ACC_COLS = 256;  // TMEM columns per accumulator buffer (2 buffers = the whole 512-column TMEM)

constexpr int CW = 32;  // epilogue chunk width in fp32 columns (one tcgen05.ld 32x32b.x32 per chunk)

// shared-memory carve-up (offsets from the 1024-aligned base): epilogue staging (EPI_WARPS x 32 rows x CW fp32 columns),
// mbarriers + TMEM slot, then the operand ring.
constexpr int SM_BARS = EPI_WARPS * 32 * CW * 4;
constexpr int SM_RING = SM_BARS + 1024;
constexpr int SM_MAX_DYNAMIC = 232448;   // 227 KB
constexpr int SM_RING_BUDGET = SM_MAX_DYNAMIC - SM_RING - 1024 /*alignment slack*/;

struct TcParams {
    void* c;
    const float* bias;
    const float* res;
    void* aux;
    int m, n, k;
    int c_dtype;
    long ldc, ldres;
    int batch2;
    long sc1, sc2;
    int a_b1, a_b2, b_b1, b_b2;  // 1 if the operand really advances along that batch level
    int a_mn, b_mn;              // operand majors (0 = K-major, 1 = MN-major)
    int n_store;                 // columns of C that are written (>= n; the extra ones see a zero accumulator)
    float alpha;
    int act;
    int accumulate;
    int split_k;
    int vec_ok;
    int epi_mode;
    int bn, stages, stage_bytes;
    int tiles_m, tiles_n, total_units;
    const bf16* dact;  // saved tensor of the activation whose derivative multiplies the result (addressed like C, row stride lddact)
    long lddact;
    float* colsum;     // colsum[b1*cs1 + b2*cs2 + n] += sum_m C[m, n]
    long cs1, cs2;
    // implicit-GEMM 3x3 stride-2 convolution over parity planes (see conv2_tc_dispatch): only the TMA producer changes
    int tma_epi;       // epilogue stores through TMA (row-per-thread math, swizzled staging, bulk tensor store / reduce-add)
    int c_b1, c_b2;    // 1 if C really advances along that batch level (TMA store coordinates)
    int conv_mode;     // 0 plain GEMM | 1 forward | 2 input gradient (one parity class) | 3 weight gradient
    int conv_kbt;      // K blocks per tap (= channels / 64)
    int conv_d;        // channels
    int conv_off[9];   // flattened (u,v) row shift of the tap: (kh >> 1) * V + (kw >> 1)
    int conv_plane[9]; // parity plane of the tap: (kh & 1) * 2 + (kw & 1)
    int conv_tap[9];   // tap id kh * 3 + kw (column block of the (co, tap, ci) weight)
    DropCfg drop;      // dropout on the output (philox.cuh); thr = 0: off
    int drop_mark;     // dropped elements of aux receive LASR_DROP_MARK (0 with aux_deriv)
    int aux_deriv;     // aux = act'(pre-activation) instead of the pre-activation (Swish)
    int epi_rot;       // 1: rotate the chunk -> epilogue-warp assignment from unit to unit (uneven chunk counts)
};


struct Unit {
    int m0, n0, b1, b2, kb_begin, num_kb;
};
__device__ __forceinline__ Unit decode_unit(const TcParams& p, int u) {
    Unit w;
    const int nb = u % p.tiles_n;
    u /= p.tiles_n;
    const int mb = u % p.tiles_m;
    u /= p.tiles_m;
    const int split = u % p.split_k, batch = u / p.split_k;
    w.m0 = mb * BM;
    w.n0 = nb * p.bn;
    w.b2 = batch % p.batch2;
    w.b1 = batch / p.batch2;
    const int total_kb = (p.k + BK - 1) / BK;
    const int kb_per = (total_kb + p.split_k - 1) / p.split_k;
    w.kb_begin = split * kb_per;
    w.num_kb = min(total_kb, w.kb_begin + kb_per) - w.kb_begin;  // <= 0 only for trailing splits: skipped by every role
    return w;
}

// ------------------------------------------------------------------------------------------------
// epilogue: one warp, one 32-row TMEM lane quarter, every (EPI_WARPS/4)-th 32-column chunk of a work unit
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
// tensor-core path only (bf16 operands): ex2/rcp approximations, ~2 ulp -- far below bf16 resolution
// sigmoid(x) = 0.5 tanh(x/2) + 0.5: ONE MUFU op (tanh.approx, rel. error ~2^-11, below bf16 resolution) instead of ex2 + rcp
__device__ __forceinline__ float sigmoid_fast(float x) {
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.5f * x));
    return fmaf(t, 0.5f, 0.5f);
}
// With h = x/2 and t = tanh(h):  swish(x) = x (1 + t)/2 = h + h t -- three instructions (MUFU included) instead of four
__device__ __forceinline__ float swish_fast(float x) {
    const float h = 0.5f * x;
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
    return fmaf(h, t, h);
}
// half_scale * 2 * swish'(x): pass half_scale = alpha / 2
__device__ __forceinline__ float dswish_scaled(float x, float half_scale) {
    // (the shorter form (1 + t + h (1 - t^2)) * half_scale with t = tanh(x/2), h = x/2 measured 4.7 % SLOWER in the FFN input-gradient
    //  GEMM: 34.4 vs 32.8 us at 9568 x 2048 x 256)
    const float r = sigmoid_fast(x);
    return (2.f * half_scale) * (r * fmaf(x, 1.f - r, 1.f));
}
__device__ __forceinline__ float dswish_fast(float x) { return dswish_scaled(x, 0.5f); }
// a = swish(x) and g = swish'(x) from ONE tanh: with h = x/2, t = tanh(h):  a = h + h t,  g = (1 + t + h (1 - t^2)) / 2
__device__ __forceinline__ void swish_and_deriv(float x, float& a, float& g) {
    const float h = 0.5f * x;
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
    a = fmaf(h, t, h);
    g = fmaf(fmaf(h, fmaf(-t, t, 1.f), t), 0.5f, 0.5f);
}
__device__ __forceinline__ float dact_fast(float saved, int act) {
    if (act == LASR_ACT_RELU) return saved > 0.f ? 1.f : 0.f;
    if (act == LASR_ACT_SWISH) return dswish_fast(saved);
    if (act == LASR_ACT_MUL) return saved;
    return 1.f;
}
__device__ __forceinline__ float act_fast(float x, int act) {
    if (act == LASR_ACT_RELU) return fmaxf(x, 0.f);
    if (act == LASR_ACT_SWISH) return swish_fast(x);
    return x;
}

// Staging buffer: 32 rows x 128 B of fp32 accumulators; the 16-byte piece `chunk` of row `row` lives at
// row * 128 + ((chunk ^ (row & 7)) << 4): conflict-free for the row-per-thread writes and the row-contiguous reads.
template <typename CT>
__device__ __forceinline__ void store4(CT* dst, const float4& f) {
    if constexpr (sizeof(CT) == 4) {
        *reinterpret_cast<float4*>(dst) = f;
    } else {
        uint2 u;
        u.x = pack_bf16x2(f.x, f.y);
        u.y = pack_bf16x2(f.z, f.w);
        *reinterpret_cast<uint2*>(dst) = u;
    }
}

// Epilogue modes: the column phase is specialised so that its inner loop carries no run-time flag tests.
enum { EPI_PLAIN = 0, EPI_RELU = 1, EPI_SWISH = 2, EPI_RES = 3, EPI_ACC = 4, EPI_GENERIC = 5, EPI_DSWISH = 6, EPI_DRELU = 7,
       EPI_DMUL = 10 };  // C = alpha * acc * saved factor (the forward pass saved act'() itself: aux_deriv)

// The staging buffer holds 32 rows x CW columns; a row is PIECES = CW/4 16-byte pieces, XOR-swizzled so that both the
// row-per-thread writes and the row-contiguous reads are bank-conflict free: piece j of row r lives at
// r*128 + ((j ^ (r & 7)) << 4).  In the column phase PIECES lanes own one row segment and a warp covers RGRP = 32 / PIECES
// rows per instruction.
template <typename CT, int MODE, bool DROP>
__device__ __forceinline__ void epilogue_unit(const TcParams& p, const Unit& w, uint32_t tmem_acc, uint8_t* stage, int q, int part,
                                              int lane) {
    constexpr int PIECES = CW / 4, RGRP = 32 / PIECES, ITERS = 32 / RGRP, ROWB = CW * 4;
    const long boff = (long)w.b1 * p.sc1 + (long)w.b2 * p.sc2;
    const int col_limit = min(p.n_store, w.n0 + p.bn);
    const int row_base = w.m0 + q * 32;
    const uint32_t taddr = tmem_acc + ((uint32_t)(q * 32) << 16);
    const int chunk = lane % PIECES, rsub = lane / PIECES;
    const int nrows = p.m - row_base - rsub;  // this lane's row RGRP*i + rsub exists iff RGRP*i < nrows
    const float alpha = p.alpha;
    CT* cbase = reinterpret_cast<CT*>(p.c) + boff;
    CT* abase = p.aux ? reinterpret_cast<CT*>(p.aux) + boff : nullptr;
    const float* rbase = p.res ? p.res + boff : nullptr;
    const bf16* dbase = p.dact ? p.dact + boff : nullptr;
    float* csbase = p.colsum ? p.colsum + (long)w.b1 * p.cs1 + (long)w.b2 * p.cs2 : nullptr;
    constexpr bool DACT = (MODE == EPI_DSWISH || MODE == EPI_DRELU || MODE == EPI_DMUL);
    uint8_t* wr = stage + lane * ROWB;
    const int wx = (lane & 7) << 4;
    // rows 4i + rsub alternate between two swizzle phases (i even / odd)
    const uint8_t* rd0 = stage + rsub * 128 + ((chunk ^ rsub) << 4);
    const uint8_t* rd1 = stage + rsub * 128 + (((chunk ^ rsub) ^ 4) << 4);
    const bool drop_on = DROP && p.drop.thr != 0;  // warp-uniform; DROP = false kernels carry none of the dropout code
    DropKey dk = {};
    if (drop_on) dk = drop_key(p.drop);
    for (int cc = part * CW; cc < p.bn; cc += CW * (EPI_WARPS / 4)) {
        const int col = w.n0 + cc + chunk * 4;  // this lane's 4 columns in the column phase
        if (w.n0 + cc >= col_limit) break;      // warp-uniform
        // vector path: whole chunks, or a partial chunk whose edge falls on a 4-column boundary (then each lane's
        // 4 columns are all inside or all outside: N = 304 score tiles, N = 4240 padded vocabularies)
        const bool fast = (MODE != EPI_GENERIC) && p.vec_ok && ((w.n0 + cc + CW <= col_limit) || (col_limit & 3) == 0);
        const bool lane_ok = col < col_limit;
        // prefetch what the column phase needs from global memory before touching TMEM
        float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
        float4 r4[ITERS];
        uint2 s2[ITERS];
        if (fast) {
            if (p.bias && lane_ok) b4 = __ldg(reinterpret_cast<const float4*>(p.bias + col));
            if constexpr (DACT) {
                const bf16* sp = dbase + (long)(row_base + rsub) * p.lddact + col;
#pragma unroll
                for (int i = 0; i < ITERS; ++i)
                    s2[i] = ldg_pred_u2(sp + (long)(RGRP * i) * p.lddact, RGRP * i < nrows && lane_ok);
            }
            if constexpr (MODE == EPI_RES) {
                const float* rp = rbase + (long)(row_base + rsub) * p.ldres + col;
#pragma unroll
                for (int i = 0; i < ITERS; ++i)
                    r4[i] = ldg_pred_f4(rp + (long)(RGRP * i) * p.ldres, RGRP * i < nrows && lane_ok);
            }
        } else if (p.bias) {
            b4.x = (col + 0 < col_limit) ? __ldg(p.bias + col + 0) : 0.f;
            b4.y = (col + 1 < col_limit) ? __ldg(p.bias + col + 1) : 0.f;
            b4.z = (col + 2 < col_limit) ? __ldg(p.bias + col + 2) : 0.f;
            b4.w = (col + 3 < col_limit) ? __ldg(p.bias + col + 3) : 0.f;
        }
        // row phase: thread = accumulator row
        {
            float v[CW];
            tc_ld32(taddr + (uint32_t)cc, v);
            __syncwarp();  // the previous chunk's column phase has finished reading the staging buffer
#pragma unroll
            for (int j = 0; j < PIECES; ++j)
                *reinterpret_cast<float4*>(wr + ((j << 4) ^ wx)) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        }
        __syncwarp();
        // column phase: PIECES lanes cover one row segment, RGRP rows per instruction
        if (fast) {
            // one running 64-bit element offset serves C and the optional pre-activation copy (same leading dimension); the
            // copy's presence and alpha == 1 are warp-uniform flags hoisted out of the loop (a nullable pointer advanced per
            // iteration costs two 64-bit selects and compares per row group)
            long off = (long)(row_base + rsub) * p.ldc + col;
            const long rstride = RGRP * p.ldc;
            const bool has_aux = abase != nullptr;
            const bool unit_alpha = alpha == 1.f;
            float4 ba = b4;
            if constexpr (MODE == EPI_PLAIN || MODE == EPI_RES) { ba.x *= alpha; ba.y *= alpha; ba.z *= alpha; ba.w *= alpha; }
            float4 cs = make_float4(0.f, 0.f, 0.f, 0.f);
            // dropout: one Philox call covers 16 columns = the four lanes of a quad (same rows, same 16-column group), so the quad
            // splits the row groups: lane t of the quad evaluates row groups i = t (mod 4) and one shuffle per row group hands every
            // lane its nibble -- ITERS / 4 calls per lane instead of ITERS
            uint32_t knib = 0xffffffffu;  // 4 keep bits per row group
            if (drop_on) {
                static_assert(ITERS % 4 == 0 && ITERS <= 8, "quad sharing of the dropout masks");
                knib = 0u;
#pragma unroll
                for (int s = 0; s < ITERS / 4; ++s) {
                    const uint32_t k16 = drop_keep16(dk, (uint32_t)(row_base + rsub + RGRP * (4 * s + (lane & 3))), (uint32_t)col >> 4);
#pragma unroll
                    for (int t = 0; t < 4; ++t)
                        knib |= ((__shfl_sync(0xffffffffu, k16, (lane & ~3) | t) >> (col & 12)) & 15u) << (4 * (4 * s + t));
                }
            }
#pragma unroll
            for (int i = 0; i < ITERS; ++i) {
                float4 f = *reinterpret_cast<const float4*>(((i & 1) ? rd1 : rd0) + i * (RGRP * ROWB));
                if (RGRP * i < nrows && lane_ok) {
                    CT* crow = cbase + off;
                    // dropout (PLAIN / RES / RELU / SWISH): one Philox call per (row, 4 columns); kx..kw = scale or 0
                    float kx = 1.f, ky = 1.f, kz = 1.f, kw = 1.f;
                    uint32_t keep4 = 15u;
                    if (drop_on) {
                        keep4 = (knib >> (4 * i)) & 15u;
                        kx = (keep4 & 1u) ? dk.scale : 0.f; ky = (keep4 & 2u) ? dk.scale : 0.f;
                        kz = (keep4 & 4u) ? dk.scale : 0.f; kw = (keep4 & 8u) ? dk.scale : 0.f;
                    }
                    if constexpr (MODE == EPI_PLAIN) {
                        f.x = fmaf(f.x, alpha, ba.x); f.y = fmaf(f.y, alpha, ba.y); f.z = fmaf(f.z, alpha, ba.z); f.w = fmaf(f.w, alpha, ba.w);
                        if (drop_on) { f.x *= kx; f.y *= ky; f.z *= kz; f.w *= kw; }
                        store4<CT>(crow, f);
                        cs.x += f.x; cs.y += f.y; cs.z += f.z; cs.w += f.w;
                    } else if constexpr (DACT) {
                        const __nv_bfloat162 h0 = *reinterpret_cast<const __nv_bfloat162*>(&s2[i].x), h1 = *reinterpret_cast<const __nv_bfloat162*>(&s2[i].y);
                        if constexpr (MODE == EPI_DSWISH) {
                            const float ha = 0.5f * alpha;
                            f.x *= dswish_scaled(__low2float(h0), ha); f.y *= dswish_scaled(__high2float(h0), ha);
                            f.z *= dswish_scaled(__low2float(h1), ha); f.w *= dswish_scaled(__high2float(h1), ha);
                        } else if constexpr (MODE == EPI_DMUL) {
                            f.x *= alpha * __low2float(h0); f.y *= alpha * __high2float(h0);
                            f.z *= alpha * __low2float(h1); f.w *= alpha * __high2float(h1);
                        } else {
                            f.x = __low2float(h0) > 0.f ? alpha * f.x : 0.f; f.y = __high2float(h0) > 0.f ? alpha * f.y : 0.f;
                            f.z = __low2float(h1) > 0.f ? alpha * f.z : 0.f; f.w = __high2float(h1) > 0.f ? alpha * f.w : 0.f;
                        }
                        store4<CT>(crow, f);
                        cs.x += f.x; cs.y += f.y; cs.z += f.z; cs.w += f.w;
                    } else if constexpr (MODE == EPI_RES) {
                        if (drop_on) {  // res + keep * scale * (alpha * acc + alpha * bias)
                            f.x = fmaf(fmaf(f.x, alpha, ba.x), kx, r4[i].x); f.y = fmaf(fmaf(f.y, alpha, ba.y), ky, r4[i].y);
                            f.z = fmaf(fmaf(f.z, alpha, ba.z), kz, r4[i].z); f.w = fmaf(fmaf(f.w, alpha, ba.w), kw, r4[i].w);
                        } else {
                            f.x = fmaf(f.x, alpha, ba.x) + r4[i].x; f.y = fmaf(f.y, alpha, ba.y) + r4[i].y;
                            f.z = fmaf(f.z, alpha, ba.z) + r4[i].z; f.w = fmaf(f.w, alpha, ba.w) + r4[i].w;
                        }
                        store4<CT>(crow, f);
                    } else if constexpr (MODE == EPI_ACC) {
                        f.x *= alpha; f.y *= alpha; f.z *= alpha; f.w *= alpha;
                        red_add_f32x4(reinterpret_cast<float*>(crow), f);
                    } else {  // EPI_RELU / EPI_SWISH (+ optional pre-activation copy)
                        f.x += b4.x; f.y += b4.y; f.z += b4.z; f.w += b4.w;
                        const bool deriv = MODE == EPI_SWISH && p.aux_deriv != 0;  // warp-uniform
                        if (has_aux && !deriv) {
                            float4 h = f;
                            if (drop_on && p.drop_mark) {
                                h.x = (keep4 & 1u) ? h.x : LASR_DROP_MARK; h.y = (keep4 & 2u) ? h.y : LASR_DROP_MARK;
                                h.z = (keep4 & 4u) ? h.z : LASR_DROP_MARK; h.w = (keep4 & 8u) ? h.w : LASR_DROP_MARK;
                            }
                            store4<CT>(abase + off, h);
                        }
                        if constexpr (MODE == EPI_RELU) {
                            f.x = fmaxf(f.x, 0.f); f.y = fmaxf(f.y, 0.f); f.z = fmaxf(f.z, 0.f); f.w = fmaxf(f.w, 0.f);
                        } else if (deriv) {
                            float4 gq;
                            swish_and_deriv(f.x, f.x, gq.x); swish_and_deriv(f.y, f.y, gq.y);
                            swish_and_deriv(f.z, f.z, gq.z); swish_and_deriv(f.w, f.w, gq.w);
                            if (drop_on && p.drop_mark) {
                                gq.x = (keep4 & 1u) ? gq.x : 0.f; gq.y = (keep4 & 2u) ? gq.y : 0.f;
                                gq.z = (keep4 & 4u) ? gq.z : 0.f; gq.w = (keep4 & 8u) ? gq.w : 0.f;
                            }
                            if (has_aux) store4<CT>(abase + off, gq);
                        } else {
                            f.x = swish_fast(f.x); f.y = swish_fast(f.y); f.z = swish_fast(f.z); f.w = swish_fast(f.w);
                        }
                        if (!unit_alpha) { f.x *= alpha; f.y *= alpha; f.z *= alpha; f.w *= alpha; }
                        if (drop_on) { f.x *= kx; f.y *= ky; f.z *= kz; f.w *= kw; }
                        store4<CT>(crow, f);
                    }
                }
                off += rstride;
            }
            if constexpr (MODE == EPI_PLAIN || DACT) {
                if (csbase) {  // warp-uniform: fold the row groups (lanes with the same piece), then one vector red per 4 columns
#pragma unroll
                    for (int o = PIECES; o < 32; o <<= 1) {
                        cs.x += __shfl_xor_sync(0xffffffffu, cs.x, o); cs.y += __shfl_xor_sync(0xffffffffu, cs.y, o);
                        cs.z += __shfl_xor_sync(0xffffffffu, cs.z, o); cs.w += __shfl_xor_sync(0xffffffffu, cs.w, o);
                    }
                    if (rsub == 0 && lane_ok) red_add_f32x4(csbase + col, cs);
                }
            }
        } else {  // ragged N edge, unaligned C or an unusual flag combination: element-wise, compact (not unrolled)
#pragma unroll 1
            for (int i = 0; i < ITERS; ++i) {
                const int row = RGRP * i + rsub;
                const int grow = row_base + row;
                const float4 f4 = *reinterpret_cast<const float4*>(stage + row * ROWB + ((chunk ^ (row & 7)) << 4));
                const float f[4] = {f4.x + b4.x, f4.y + b4.y, f4.z + b4.z, f4.w + b4.w};
                if (grow >= p.m) continue;
#pragma unroll 1
                for (int e = 0; e < 4; ++e) {
                    if (col + e >= col_limit) break;
                    const long off = (long)grow * p.ldc + col + e;
                    if (p.accumulate) {
                        atomicAdd(reinterpret_cast<float*>(cbase + off), alpha * f[e]);
                    } else {
                        float x;
                        if (dbase) {
                            x = alpha * f[e] * dact_fast(__bfloat162float(dbase[(long)grow * p.lddact + col + e]), p.act);
                        } else {
                            const bool keep = !drop_on || drop_keep1(dk, (uint32_t)grow, (uint32_t)(col + e));
                            if (abase) {
                                if (p.aux_deriv) abase[off] = from_f32<CT>((keep || !p.drop_mark) ? dswish_fast(f[e]) : 0.f);
                                else abase[off] = from_f32<CT>((keep || !p.drop_mark) ? f[e] : LASR_DROP_MARK);
                            }
                            x = alpha * act_fast(f[e], p.act);
                            if (drop_on) x = keep ? x * dk.scale : 0.f;
                            if (rbase) x += rbase[(long)grow * p.ldres + col + e];
                        }
                        cbase[off] = from_f32<CT>(x);
                        if (csbase) atomicAdd(csbase + col + e, x);
                    }
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// TMA-store epilogue of the PLAIN / RELU / SWISH / ACC modes without colsum (whenever C / aux / bias meet the 16-byte
// alignment rules: setup_tma_epilogue).
// The accumulator row a thread reads from TMEM (32 consecutive columns) is finished IN PLACE -- bias as warp-uniform float4
// loads -- converted, written to a swizzled 32 x 32 staging box
// (SWIZZLE_64B for bf16, SWIZZLE_128B for fp32: the same XOR patterns that make the row-per-thread 16-byte stores conflict
// free) and handed to ONE bulk tensor store (or reduce-add) per box.  Compared with the register -> smem -> register ->
// global column phase this removes every LDS, STG, 64-bit address computation and edge predicate from the 16 epilogue warps
// (the FFN fc1 + Swish kernel was issue-bound: 59 % issue-slot utilisation, 58 % LSU wavefronts, tensor pipe 21 %); the TMA
// unit clips rows >= M and columns >= N, so ragged shapes (N = 299, V = 4233) take the same path.
// ------------------------------------------------------------------------------------------------
template <typename CT, int MODE, bool DROP>
__device__ __forceinline__ void epilogue_unit_tma(const TcParams& p, const Unit& w, uint32_t tmem_acc, uint8_t* stage, int q, int part,
                                                  int lane, const CUtensorMap* mc, const CUtensorMap* mx, int& buf) {
    constexpr bool BF = sizeof(CT) == 2;
    const int col_limit = min(p.n_store, w.n0 + p.bn);
    const int row0 = w.m0 + q * 32, row = row0 + lane;
    const uint32_t taddr = tmem_acc + ((uint32_t)(q * 32) << 16);
    const float alpha = p.alpha;
    const bool has_aux = p.aux != nullptr;   // warp-uniform
    const bool dbl = BF && !has_aux;         // two 2 KB boxes alternate; otherwise one 4 KB set (C, or C + aux)
    const int cb1 = w.b1 * p.c_b1, cb2 = w.b2 * p.c_b2;
    const bool drop_on = DROP && p.drop.thr != 0;  // warp-uniform
    DropKey dk = {};
    if (drop_on) dk = drop_key(p.drop);
    const float alpha_s = drop_on ? alpha * dk.scale : alpha;  // 1 / (1 - p) rides on alpha
    for (int cc = part * 32; cc < p.bn; cc += 32 * (EPI_WARPS / 4)) {
        const int col0 = w.n0 + cc;
        if (col0 >= col_limit) break;  // warp-uniform
        const bool full = col0 + 32 <= col_limit;
        // dropout: the keep masks of this thread's 32-column row segment are evaluated between the ISSUE of the TMEM load and
        // its wait: they depend on nothing the accumulator holds, so the Philox latency chain hides behind the load's
        // (two calls: packed 0xffff / 0 lane masks, mk[t] = columns col0 + 2t and col0 + 2t + 1 -- philox.cuh)
        uint32_t mk[16];
        float v[32];
        if constexpr (DROP) {
            tc_ld32_issue(taddr + (uint32_t)cc, v);
            if (drop_on) {
                uint32_t h0[8], h1[8];
                drop_masks16(dk, (uint32_t)row, (uint32_t)col0 >> 4, h0);
                drop_masks16(dk, (uint32_t)row, ((uint32_t)col0 >> 4) + 1u, h1);
#pragma unroll
                for (int t = 0; t < 8; ++t) { mk[t] = h0[t]; mk[8 + t] = h1[t]; }
            }
            tc_ld_wait32(v);
        } else {
            tc_ld32(taddr + (uint32_t)cc, v);
        }
        // ---- finish the row in place
        if constexpr (MODE == EPI_ACC) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] *= alpha;
        } else {
            // bias: the same 32 floats for every lane (warp-uniform 16-byte loads, L1-resident), consumed quad by quad
            const bool has_bias = p.bias != nullptr;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
                if (has_bias) {
                    const int c = col0 + 4 * j;
                    if (full) {
                        b = __ldg(reinterpret_cast<const float4*>(p.bias + c));
                    } else {
                        b.x = c + 0 < col_limit ? __ldg(p.bias + c + 0) : 0.f;
                        b.y = c + 1 < col_limit ? __ldg(p.bias + c + 1) : 0.f;
                        b.z = c + 2 < col_limit ? __ldg(p.bias + c + 2) : 0.f;
                        b.w = c + 3 < col_limit ? __ldg(p.bias + c + 3) : 0.f;
                    }
                }
                if constexpr (MODE == EPI_PLAIN) {
                    v[4 * j] = fmaf(v[4 * j], alpha_s, alpha_s * b.x); v[4 * j + 1] = fmaf(v[4 * j + 1], alpha_s, alpha_s * b.y);
                    v[4 * j + 2] = fmaf(v[4 * j + 2], alpha_s, alpha_s * b.z); v[4 * j + 3] = fmaf(v[4 * j + 3], alpha_s, alpha_s * b.w);
                    if (drop_on) {  // dropped -> +0
                        v[4 * j] = drop_and(v[4 * j], drop_mask_lo(mk[2 * j])); v[4 * j + 1] = drop_and(v[4 * j + 1], drop_mask_hi(mk[2 * j]));
                        v[4 * j + 2] = drop_and(v[4 * j + 2], drop_mask_lo(mk[2 * j + 1])); v[4 * j + 3] = drop_and(v[4 * j + 3], drop_mask_hi(mk[2 * j + 1]));
                    }
                } else {  // EPI_RELU / EPI_SWISH: pre-activation = acc + bias
                    v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
                }
            }
        }
        // ---- staging box free?  (only lane 0 issues bulk stores, so only lane 0 has groups to wait for)
        // (Doing the Swish / Swish' math of the chunk BEFORE this wait, with the packed derivative held in 16 registers across it,
        //  measured slower: fc1 with dropout 105.6 vs 91.7 us at C2 / B = 126 -- 52 bytes of spills at the 96-register cap.)
        uint8_t* sb = stage + (dbl ? buf * 2048 : 0);
        if (lane == 0) {
            if (dbl) bulk_wait_read<1>();
            else bulk_wait_read<0>();
        }
        __syncwarp();
        if constexpr (MODE == EPI_RELU || MODE == EPI_SWISH) {
            const bool deriv = MODE == EPI_SWISH && has_aux && p.aux_deriv != 0;  // warp-uniform
            const bool hmask = drop_on && p.drop_mark;  // warp-uniform: the saved tensor carries the mask
            if (deriv) {  // aux = swish'(h) (0 where dropped) and v = swish(h), 8 columns at a time (one tanh serves both)
                uint8_t* sx = stage + 2048;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float gq[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) swish_and_deriv(v[8 * j + e], v[8 * j + e], gq[e]);
                    uint4 u;
                    u.x = pack_bf16x2(gq[0], gq[1]); u.y = pack_bf16x2(gq[2], gq[3]);
                    u.z = pack_bf16x2(gq[4], gq[5]); u.w = pack_bf16x2(gq[6], gq[7]);
                    if (hmask) { u.x &= mk[4 * j]; u.y &= mk[4 * j + 1]; u.z &= mk[4 * j + 2]; u.w &= mk[4 * j + 3]; }
                    *reinterpret_cast<uint4*>(sx + lane * 64 + ((j ^ ((lane >> 1) & 3)) << 4)) = u;
                }
            } else if (has_aux) {  // pre-activation copy (bf16 on this path); dropped elements carry the marker whose act'() is 0
                uint8_t* sx = stage + 2048;
                const uint32_t mark2 = pack_bf16x2(LASR_DROP_MARK, LASR_DROP_MARK);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    uint4 u;
                    u.x = pack_bf16x2(v[8 * j], v[8 * j + 1]); u.y = pack_bf16x2(v[8 * j + 2], v[8 * j + 3]);
                    u.z = pack_bf16x2(v[8 * j + 4], v[8 * j + 5]); u.w = pack_bf16x2(v[8 * j + 6], v[8 * j + 7]);
                    if (hmask) {
                        u.x = (u.x & mk[4 * j]) | (mark2 & ~mk[4 * j]); u.y = (u.y & mk[4 * j + 1]) | (mark2 & ~mk[4 * j + 1]);
                        u.z = (u.z & mk[4 * j + 2]) | (mark2 & ~mk[4 * j + 2]); u.w = (u.w & mk[4 * j + 3]) | (mark2 & ~mk[4 * j + 3]);
                    }
                    *reinterpret_cast<uint4*>(sx + lane * 64 + ((j ^ ((lane >> 1) & 3)) << 4)) = u;
                }
            }
            if (!deriv) {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = (MODE == EPI_RELU) ? fmaxf(v[j], 0.f) : swish_fast(v[j]);
            }
            if (alpha_s != 1.f) {  // warp-uniform: no multiply on the alpha == 1, p == 0 path
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] *= alpha_s;
            }
            if constexpr (!BF) {  // fp32 result: mask the values; the bf16 result is masked after packing (one AND per pair)
                if (drop_on) {
#pragma unroll
                    for (int t = 0; t < 16; ++t) { v[2 * t] = drop_and(v[2 * t], drop_mask_lo(mk[t])); v[2 * t + 1] = drop_and(v[2 * t + 1], drop_mask_hi(mk[t])); }
                }
            }
        }
        if constexpr (BF) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                uint4 u;
                u.x = pack_bf16x2(v[8 * j], v[8 * j + 1]); u.y = pack_bf16x2(v[8 * j + 2], v[8 * j + 3]);
                u.z = pack_bf16x2(v[8 * j + 4], v[8 * j + 5]); u.w = pack_bf16x2(v[8 * j + 6], v[8 * j + 7]);
                if constexpr (MODE == EPI_RELU || MODE == EPI_SWISH) {
                    if (drop_on) { u.x &= mk[4 * j]; u.y &= mk[4 * j + 1]; u.z &= mk[4 * j + 2]; u.w &= mk[4 * j + 3]; }
                }
                *reinterpret_cast<uint4*>(sb + lane * 64 + ((j ^ ((lane >> 1) & 3)) << 4)) = u;
            }
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j)
                *reinterpret_cast<float4*>(sb + lane * 128 + ((j ^ (lane & 7)) << 4)) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
            if constexpr (MODE == EPI_ACC) tma_reduce_add_4d(mc, sb, col0, row0, cb2, cb1);
            else tma_store_4d(mc, sb, col0, row0, cb2, cb1);
            if constexpr (MODE == EPI_RELU || MODE == EPI_SWISH) {
                if (has_aux) tma_store_4d(mx, stage + 2048, col0, row0, cb2, cb1);
            }
            bulk_commit();
        }
        if (dbl) buf ^= 1;
    }
}

// MODE / C_F32 specialise the epilogue warps (one kernel per epilogue keeps the instruction footprint and the register
// allocation of each variant minimal); operand majors are run-time values: they only steer the two single-thread roles.
// The three roles walk the same work units: blockIdx.x, + gridDim.x, ... of the (batch, split, m, n) list; a unit with no
// K blocks (a trailing split) is skipped by every role.
template <int MODE, bool C_F32, bool DROP>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
               const __grid_constant__ CUtensorMap tma_c, const __grid_constant__ CUtensorMap tma_x, const TcParams p) {
    const bool A_MN = p.a_mn != 0, B_MN = p.b_mn != 0;
    extern __shared__ uint8_t smem_raw[];
    // align inside the shared window (keeps the address space visible to the compiler: LDS/STS, not generic LD/ST)
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + SM_BARS);
    uint64_t* empty_bar = full_bar + MAX_STAGES;
    uint64_t* acc_full = empty_bar + MAX_STAGES;
    uint64_t* acc_empty = acc_full + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
    uint8_t* ring = smem + SM_RING;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&tma_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&tma_b) : "memory");
        if (p.tma_epi) {
            asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&tma_c) : "memory");
            if (p.aux) asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&tma_x) : "memory");
        }
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < MAX_STAGES; ++s) {
            mbar_init(full_bar + s, 1);
            mbar_init(empty_bar + s, 1);
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(acc_full + s, 1);
            mbar_init(acc_empty + s, EPI_WARPS);  // one arrival per epilogue warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"((uint32_t)(2 * ACC_COLS))
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
    // Programmatic dependent launch: everything above (barrier init, TMEM allocation, tensor-map prefetch) touches no global
    // data and may overlap the tail of the previous kernel in the stream; from here on the roles read and write global memory.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");

    if (warp == 0) {
        if (lane == 0) {
            int s = 0;
            uint32_t ph = 0;
            for (int u = blockIdx.x; u < p.total_units; u += gridDim.x) {
                const Unit w = decode_unit(p, u);
                if (w.num_kb <= 0) continue;
                const int ab1 = w.b1 * p.a_b1, ab2 = w.b2 * p.a_b2, bb1 = w.b1 * p.b_b1, bb2 = w.b2 * p.b_b2;
                for (int i = 0; i < w.num_kb; ++i) {
                    mbar_wait(empty_bar + s, ph ^ 1);
                    mbar_arrive_expect_tx(full_bar + s, (uint32_t)p.stage_bytes);
                    uint8_t* sa = ring + s * p.stage_bytes;
                    uint8_t* sb = sa + A_BYTES;
                    const int k0 = (w.kb_begin + i) * BK;
                    if (p.conv_mode != 0) {
                        const int kb = w.kb_begin + i;
                        if (p.conv_mode == 1) {         // A = h1 planes (rows shifted per tap), B = (co, tap*ci) weight, both K-major
                            const int tp = kb / p.conv_kbt, kc = kb - tp * p.conv_kbt;
                            tma_load_4d(sa, &tma_a, full_bar + s, kc * BK, w.m0 + p.conv_off[tp], p.conv_plane[tp], w.b1);
                            tma_load_4d(sb, &tma_b, full_bar + s, k0, w.n0, 0, 0);
                        } else if (p.conv_mode == 2) {  // A = dY (K-major, rows shifted back), B = weight MN-major at the tap's columns
                            const int tp = kb / p.conv_kbt, kc = kb - tp * p.conv_kbt;
                            tma_load_4d(sa, &tma_a, full_bar + s, kc * BK, w.m0 - p.conv_off[tp], 0, w.b1);
                            for (int j = 0; j < p.bn / 64; ++j)
                                tma_load_4d(sb + j * 8192, &tma_b, full_bar + s, w.n0 + 64 * j + p.conv_tap[tp] * p.conv_d, kc * BK, 0, 0);
                        } else {                        // A = dY^T, B = h1 planes, both MN-major; the N tile selects the tap
                            const int tp = w.n0 / p.conv_d, nloc = w.n0 - tp * p.conv_d;
#pragma unroll
                            for (int j = 0; j < BM / 64; ++j)
                                tma_load_4d(sa + j * 8192, &tma_a, full_bar + s, w.m0 + 64 * j, k0, 0, w.b1);
                            for (int j = 0; j < p.bn / 64; ++j)
                                tma_load_4d(sb + j * 8192, &tma_b, full_bar + s, nloc + 64 * j, k0 + p.conv_off[tp], p.conv_plane[tp], w.b1);
                        }
                    } else {
                        if (!A_MN) {
                            tma_load_4d(sa, &tma_a, full_bar + s, k0, w.m0, ab2, ab1);  // box {64 k, 128 m}
                        } else {
#pragma unroll
                            for (int j = 0; j < BM / 64; ++j)  // box {64 m, 64 k}
                                tma_load_4d(sa + j * 8192, &tma_a, full_bar + s, w.m0 + 64 * j, k0, ab2, ab1);
                        }
                        if (!B_MN) {
                            tma_load_4d(sb, &tma_b, full_bar + s, k0, w.n0, bb2, bb1);  // box {64 k, BN n}
                        } else {
                            for (int j = 0; j < p.bn / 64; ++j)
                                tma_load_4d(sb + j * 8192, &tma_b, full_bar + s, w.n0 + 64 * j, k0, bb2, bb1);
                        }
                    }
                    if (++s == p.stages) { s = 0; ph ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // instruction descriptor (cute::UMMA::InstrDescriptor): c=f32, a=b=bf16, majors, N>>3, M>>4
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((A_MN ? 1u : 0u) << 15) | ((B_MN ? 1u : 0u) << 16) |
                                   ((uint32_t)(p.bn >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
            int s = 0, as = 0;
            uint32_t ph = 0, aph = 0;
            for (int u = blockIdx.x; u < p.total_units; u += gridDim.x) {
                const Unit w = decode_unit(p, u);
                if (w.num_kb <= 0) continue;
                mbar_wait(acc_empty + as, aph ^ 1);  // the epilogue has drained this accumulator buffer
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + (uint32_t)(as * ACC_COLS);
                for (int i = 0; i < w.num_kb; ++i) {
                    mbar_wait(full_bar + s, ph);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(ring + s * p.stage_bytes);
                    const uint32_t sb = sa + A_BYTES;
#pragma unroll
                    for (int kk = 0; kk < BK / UMMA_K; ++kk) {
                        // K-major: +32 B per UMMA_K inside the 128 B swizzle row; SBO = 8 rows * 128 B.
                        // MN-major: +16 K-rows * 128 B; LBO = next 64-wide MN atom (64 K-rows * 128 B), SBO = 8 K-rows.
                        const uint64_t da = A_MN ? umma_desc(sa + kk * 2048, 8192, 1024) : umma_desc(sa + kk * 32, 16, 1024);
                        const uint64_t db = B_MN ? umma_desc(sb + kk * 2048, 8192, 1024) : umma_desc(sb + kk * 32, 16, 1024);
                        tc_mma_bf16(tmem_d, da, db, idesc, (i > 0 || kk > 0) ? 1u : 0u);
                    }
                    tc_commit(empty_bar + s);  // frees the smem slot once these MMAs retire
                    if (++s == p.stages) { s = 0; ph ^= 1; }
                }
                tc_commit(acc_full + as);
                if ((as ^= 1) == 0) aph ^= 1;
            }
        }
    } else {
        const int q = warp & 3;           // TMEM lane quarter this warp may access
        const int ew = warp - 2;          // private staging slice
        const int part = ew >> 2;         // which CW-column chunks of the tile (chunk index % (EPI_WARPS/4))
        uint8_t* stage = smem + ew * (32 * CW * 4);
        int as = 0, sbuf = 0;
        uint32_t aph = 0;
        typedef typename std::conditional<C_F32, float, bf16>::type CT;
        constexpr bool TMA_OK = MODE == EPI_PLAIN || MODE == EPI_RELU || MODE == EPI_SWISH || MODE == EPI_ACC;  // setup_tma_epilogue
        const bool tma_epi = TMA_OK && p.tma_epi != 0;
        // N tiles whose 32-column chunks do not divide evenly among the four warps of a lane quarter (BN = 160: 5 chunks) leave one
        // warp with twice the work of the others in EVERY unit; rotating the chunk -> warp assignment from unit to unit spreads it
        // (the two accumulator buffers let a warp run one unit ahead of the slowest one)
        int urot = 0;
        for (int u = blockIdx.x; u < p.total_units; u += gridDim.x) {
            const Unit w = decode_unit(p, u);
            if (w.num_kb <= 0) continue;
            mbar_wait(acc_full + as, aph);  // (sleeping between polls, 32-300 ns, changes nothing: the spin is not what limits the epilogue)
            tc_fence_after();
            const uint32_t tmem_acc = tmem_base + (uint32_t)(as * ACC_COLS);
            const int part_u = (part + urot) & (EPI_WARPS / 4 - 1);
            urot += p.epi_rot;
            if constexpr (TMA_OK) {
                if (tma_epi) epilogue_unit_tma<CT, MODE, DROP>(p, w, tmem_acc, stage, q, part_u, lane, &tma_c, &tma_x, sbuf);
                else epilogue_unit<CT, MODE, DROP>(p, w, tmem_acc, stage, q, part_u, lane);
            } else {
                epilogue_unit<CT, MODE, DROP>(p, w, tmem_acc, stage, q, part_u, lane);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(acc_empty + as);
            if ((as ^= 1) == 0) aph ^= 1;
        }
        if (tma_epi && lane == 0) bulk_wait_read<0>();  // the staging boxes must outlive the bulk stores that read them
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)(2 * ACC_COLS))
                     : "memory");
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static PFN_cuTensorMapEncodeTiled_v12000 get_encode() {
    static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
    }
    return fn;
}

static int sm_count() {
    static int n = 0;
    if (!n) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
            n = 148;
    }
    return n;
}

// operand stored row-major as (outer rows, inner contiguous) with row stride ld (elements), two batch levels.
static int make_map(CUtensorMap* map, const void* base, long inner, long rows, long ld, int nb2, long s2, int nb1, long s1,
                    int box_inner, int box_rows) {
    auto enc = get_encode();
    if (!enc) {
        set_error("cuTensorMapEncodeTiled entry point unavailable");
        return LASR_ERR_DRIVER;
    }
    const bool use2 = (s2 != 0 && nb2 > 1), use1 = (s1 != 0 && nb1 > 1);
    cuuint64_t dims[4] = {(cuuint64_t)inner, (cuuint64_t)rows, (cuuint64_t)(use2 ? nb2 : 1), (cuuint64_t)(use1 ? nb1 : 1)};
    const cuuint64_t row_bytes = (cuuint64_t)ld * 2;
    cuuint64_t strides[3] = {row_bytes, use2 ? (cuuint64_t)s2 * 2 : row_bytes, use1 ? (cuuint64_t)s1 * 2 : row_bytes};
    cuuint32_t box[4] = {(cuuint32_t)box_inner, (cuuint32_t)box_rows, 1, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (strides[0] & 15) || (strides[1] & 15) || (strides[2] & 15)) {
        set_error("gemm_tc: operand base/strides must be 16-byte aligned (base=%p ld=%ld s2=%ld s1=%ld)", base, ld, s2, s1);
        return LASR_ERR_BAD_ARG;
    }
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed (%d): inner=%ld rows=%ld ld=%ld", (int)r, inner, rows, ld);
        return LASR_ERR_DRIVER;
    }
    return LASR_OK;
}

// C (or the pre-activation copy) as a TMA store target: 32 x 32 boxes, SWIZZLE_64B for bf16 rows (64 B) and SWIZZLE_128B for
// fp32 rows (128 B).  Returns 1 if the tensor cannot be described (alignment): the caller then keeps the register epilogue.
static int make_store_map(CUtensorMap* map, const void* base, int dtype, long cols, long rows, long ld, int nb2, long s2, int nb1,
                          long s1) {
    auto enc = get_encode();
    if (!enc || !base) return 1;
    const long es = dtype == LASR_F32 ? 4 : 2;
    const bool use2 = (s2 != 0 && nb2 > 1), use1 = (s1 != 0 && nb1 > 1);
    cuuint64_t dims[4] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)(use2 ? nb2 : 1), (cuuint64_t)(use1 ? nb1 : 1)};
    const cuuint64_t row_bytes = (cuuint64_t)ld * es;
    cuuint64_t strides[3] = {row_bytes, use2 ? (cuuint64_t)s2 * es : row_bytes, use1 ? (cuuint64_t)s1 * es : row_bytes};
    cuuint32_t box[4] = {32, 32, 1, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (strides[0] & 15) || (strides[1] & 15) || (strides[2] & 15)) return 1;
    CUresult r = enc(map, dtype == LASR_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4,
                     const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     dtype == LASR_F32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : 1;
}

// Decide whether the TMA-store epilogue applies and build its maps (C and, if present, the pre-activation copy).
static void setup_tma_epilogue(TcParams& p, CUtensorMap* mc, CUtensorMap* mx, int nb1, int nb2) {
    memset(mc, 0, sizeof(*mc));
    memset(mx, 0, sizeof(*mx));
    p.tma_epi = 0;
    p.c_b1 = (p.sc1 != 0 && nb1 > 1);
    p.c_b2 = (p.sc2 != 0 && nb2 > 1);
    // Row-per-thread math makes the residual / saved-activation reads 32-lines-per-instruction gathers and the column sums a
    // 31-shuffle transpose: measured slower than the column-phase epilogue (fc2 + residual 62 vs 51 us, dswish + colsum 128 vs
    // 103 us at C2/B=126), so RES, the dact modes, colsum and GENERIC keep it (TMA_OK in gemm_tc_kernel).
    if (!(p.epi_mode == EPI_PLAIN || p.epi_mode == EPI_RELU || p.epi_mode == EPI_SWISH || p.epi_mode == EPI_ACC) || p.colsum) return;
    // bulk tensor stores clip at 16-byte granularity (measured: tools/tma_clip_probe.py): a row whose last 16-byte chunk is
    // partial would get zeros written past column n_store, so ragged widths keep the register epilogue
    if (((long)p.n_store * (p.c_dtype == LASR_F32 ? 4 : 2)) & 15) return;
    if (p.aux && p.c_dtype == LASR_F32) return;                        // the staging set holds C + aux only for bf16
    if (p.bias && (reinterpret_cast<uintptr_t>(p.bias) & 15)) return;
    if (make_store_map(mc, p.c, p.c_dtype, p.n_store, p.m, p.ldc, nb2, p.sc2, nb1, p.sc1)) return;
    if (p.aux && make_store_map(mx, p.aux, p.c_dtype, p.n_store, p.m, p.ldc, nb2, p.sc2, nb1, p.sc1)) return;
    p.tma_epi = 1;
}

// N-tile width: a multiple of `gran` (16 for K-major B, 64 for MN-major B) up to 256 that wastes the fewest padded
// columns; ties go to the wider tile (fewer A re-reads, fewer epilogue tails).
static int pick_bn(int n, int gran) {
    if (n <= 256) return (n + gran - 1) / gran * gran;
    int best = 256;
    long best_pad = (long)((n + 255) / 256) * 256;
    for (int bn = 256 - gran; bn >= 128; bn -= gran) {
        const long pad = (long)((n + bn - 1) / bn) * bn;
        if (pad < best_pad) { best = bn; best_pad = pad; }
    }
    return best;
}

typedef void (*TcKernel)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const TcParams);

template <int MODE, bool C_F32, bool DROP = false>
static TcKernel configured_kernel() {
    static bool configured = false;
    TcKernel k = gemm_tc_kernel<MODE, C_F32, DROP>;
    if (!configured) {
        if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_MAX_DYNAMIC) != cudaSuccess) return nullptr;
        configured = true;
    }
    return k;
}

static TcKernel pick_kernel(int mode, bool f32) {
    if (f32) {
        switch (mode) {
            case EPI_PLAIN: return configured_kernel<EPI_PLAIN, true>();
            case EPI_RELU: return configured_kernel<EPI_RELU, true>();
            case EPI_SWISH: return configured_kernel<EPI_SWISH, true>();
            case EPI_RES: return configured_kernel<EPI_RES, true>();
            case EPI_ACC: return configured_kernel<EPI_ACC, true>();
            case EPI_DSWISH: return configured_kernel<EPI_DSWISH, true>();
            case EPI_DRELU: return configured_kernel<EPI_DRELU, true>();
            case EPI_DMUL: return configured_kernel<EPI_DMUL, true>();
            default: return configured_kernel<EPI_GENERIC, true>();
        }
    }
    switch (mode) {
        case EPI_PLAIN: return configured_kernel<EPI_PLAIN, false>();
        case EPI_RELU: return configured_kernel<EPI_RELU, false>();
        case EPI_SWISH: return configured_kernel<EPI_SWISH, false>();
        case EPI_DSWISH: return configured_kernel<EPI_DSWISH, false>();
        case EPI_DRELU: return configured_kernel<EPI_DRELU, false>();
        case EPI_DMUL: return configured_kernel<EPI_DMUL, false>();
        default: return configured_kernel<EPI_GENERIC, false>();
    }
}

// dropout variants: separate instantiations, so that the p = 0 kernels are the round-1 kernels
static TcKernel pick_drop_kernel(int mode, bool f32) {
    if (f32) {
        switch (mode) {
            case EPI_PLAIN: return configured_kernel<EPI_PLAIN, true, true>();
            case EPI_RELU: return configured_kernel<EPI_RELU, true, true>();
            case EPI_SWISH: return configured_kernel<EPI_SWISH, true, true>();
            case EPI_RES: return configured_kernel<EPI_RES, true, true>();
            default: return configured_kernel<EPI_GENERIC, true, true>();
        }
    }
    switch (mode) {
        case EPI_PLAIN: return configured_kernel<EPI_PLAIN, false, true>();
        case EPI_RELU: return configured_kernel<EPI_RELU, false, true>();
        case EPI_SWISH: return configured_kernel<EPI_SWISH, false, true>();
        default: return configured_kernel<EPI_GENERIC, false, true>();
    }
}

static int launch_tc(const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mc, const CUtensorMap& mx, const TcParams& p,
                     cudaStream_t st) {
    const bool f32 = p.c_dtype == LASR_F32;
    TcKernel kern;
    if (p.drop.thr != 0) {
        if (p.epi_mode == EPI_ACC || p.epi_mode == EPI_DSWISH || p.epi_mode == EPI_DRELU || p.epi_mode == EPI_DMUL) {
            set_error("gemm_tc: dropout is not available with this epilogue");
            return LASR_ERR_UNSUPPORTED;
        }
        kern = pick_drop_kernel(p.epi_mode, f32);
    } else {
        kern = pick_kernel(p.epi_mode, f32);
    }
    if (!kern) return check_launch("gemm_tc smem attr");
    const int smem_bytes = SM_RING + p.stages * p.stage_bytes + 1024;
    const int grid = p.total_units < sm_count() ? p.total_units : sm_count();
    static int pdl = -1;  // LASR_PDL=0: developer switch
    if (pdl < 0) { const char* e = getenv("LASR_PDL"); pdl = e ? atoi(e) : 1; }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(GEMM_THREADS);
    cfg.dynamicSmemBytes = smem_bytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    if (cudaLaunchKernelEx(&cfg, kern, ma, mb, mc, mx, p) != cudaSuccess) return check_launch("gemm_tc launch");
    return check_launch("gemm_tc");
}

int gemm_tc_dispatch(const lasr_gemm_args* a, cudaStream_t st) {
    const int n_store = a->n_store ? a->n_store : a->n;
    // N tiles are multiples of 32 columns: the TMA-store epilogue writes whole 32-column boxes, clipped only at the tensor edge
    const int gran = a->trans_b ? 64 : 32;
    int bn = pick_bn(n_store, gran);
    // Few row tiles (the decoder: 126 x 41 = 5166 rows = 41 tiles for 148 SMs): narrower N tiles until the work units cover at
    // least half of the SMs -- the A tile is re-read from L2 by more units, but a unit then takes proportionally less time
    // and 41-unit launches ran on 28 % of the machine.
    const long per_n = (long)ceil_div(a->m, BM) * (a->split_k < 1 ? 1 : a->split_k) * a->batch1 * a->batch2;
    while (per_n * ceil_div(n_store, bn) * 2 <= sm_count() && bn % (2 * gran) == 0 && bn / 2 >= 64) bn /= 2;
    CUtensorMap ma, mb;
    int rc;
    if (!a->trans_a) rc = make_map(&ma, a->a, a->k, a->m, a->lda, a->batch2, a->sa2, a->batch1, a->sa1, BK, BM);
    else rc = make_map(&ma, a->a, a->m, a->k, a->lda, a->batch2, a->sa2, a->batch1, a->sa1, 64, BK);
    if (rc) return rc;
    if (!a->trans_b) rc = make_map(&mb, a->b, a->k, a->n, a->ldb, a->batch2, a->sb2, a->batch1, a->sb1, BK, bn);
    else rc = make_map(&mb, a->b, a->n, a->k, a->ldb, a->batch2, a->sb2, a->batch1, a->sb1, 64, BK);
    if (rc) return rc;
    if (a->res && a->c_dtype != LASR_F32) {
        set_error("gemm_tc: a residual needs an fp32 C");
        return LASR_ERR_UNSUPPORTED;
    }

    TcParams p;
    p.c = a->c; p.bias = a->bias; p.res = a->res; p.aux = a->aux;
    p.m = a->m; p.n = a->n; p.k = a->k; p.c_dtype = a->c_dtype;
    p.ldc = a->ldc; p.ldres = a->ldres; p.batch2 = a->batch2; p.sc1 = a->sc1; p.sc2 = a->sc2;
    p.a_b1 = (a->sa1 != 0 && a->batch1 > 1); p.a_b2 = (a->sa2 != 0 && a->batch2 > 1);
    p.b_b1 = (a->sb1 != 0 && a->batch1 > 1); p.b_b2 = (a->sb2 != 0 && a->batch2 > 1);
    p.alpha = a->alpha; p.act = a->act; p.accumulate = a->accumulate; p.split_k = a->split_k < 1 ? 1 : a->split_k;
    const long esz = a->c_dtype == LASR_F32 ? 4 : 2;
    auto al16 = [&](long elems, long es) { return ((elems * es) & 15) == 0; };
    p.vec_ok = ((reinterpret_cast<uintptr_t>(a->c) & 15) == 0) && al16(a->ldc, esz) && al16(a->sc1, esz) && al16(a->sc2, esz);
    if (a->aux) p.vec_ok = p.vec_ok && ((reinterpret_cast<uintptr_t>(a->aux) & 15) == 0);
    if (a->bias) p.vec_ok = p.vec_ok && ((reinterpret_cast<uintptr_t>(a->bias) & 15) == 0);
    if (a->res) p.vec_ok = p.vec_ok && ((reinterpret_cast<uintptr_t>(a->res) & 15) == 0) && al16(a->ldres, 4);
    p.dact = reinterpret_cast<const bf16*>(a->dact); p.lddact = a->lddact;
    p.colsum = a->colsum; p.cs1 = a->cs1; p.cs2 = a->cs2;
    if (a->dact) p.vec_ok = p.vec_ok && ((reinterpret_cast<uintptr_t>(a->dact) & 7) == 0) && ((a->lddact * 2) % 8 == 0) && al16(a->sc1, 2) && al16(a->sc2, 2);
    if (a->colsum) p.vec_ok = p.vec_ok && ((reinterpret_cast<uintptr_t>(a->colsum) & 15) == 0) && al16(a->cs1, 4) && al16(a->cs2, 4);
    p.drop.state = reinterpret_cast<const unsigned long long*>(a->drop_state);
    p.drop.site = a->drop_site; p.drop.thr = a->drop_thr; p.drop.scale = a->drop_scale;
    p.drop_mark = a->drop_mark_aux;
    p.aux_deriv = a->aux_deriv;
    p.epi_rot = ((bn + 31) / 32) % (EPI_WARPS / 4) != 0 ? 1 : 0;
    if (a->accumulate) p.epi_mode = EPI_ACC;
    else if (a->dact && a->act == LASR_ACT_SWISH) p.epi_mode = EPI_DSWISH;
    else if (a->dact && a->act == LASR_ACT_RELU) p.epi_mode = EPI_DRELU;
    else if (a->dact && a->act == LASR_ACT_MUL) p.epi_mode = EPI_DMUL;
    else if (a->colsum && (a->res || a->aux || a->act != LASR_ACT_NONE)) p.epi_mode = EPI_GENERIC;
    else if (a->res && a->act == LASR_ACT_NONE && !a->aux) p.epi_mode = EPI_RES;
    else if (!a->res && a->act == LASR_ACT_RELU) p.epi_mode = EPI_RELU;
    else if (!a->res && a->act == LASR_ACT_SWISH) p.epi_mode = EPI_SWISH;
    else if (!a->res && !a->aux && a->act == LASR_ACT_NONE) p.epi_mode = EPI_PLAIN;
    else p.epi_mode = EPI_GENERIC;
    p.bn = bn;
    p.stage_bytes = A_BYTES + bn * BK * 2;
    p.stages = SM_RING_BUDGET / p.stage_bytes;
    if (p.stages > MAX_STAGES) p.stages = MAX_STAGES;
    p.tiles_m = ceil_div(a->m, BM);
    p.tiles_n = ceil_div(n_store, bn);
    p.n_store = n_store;
    const long units = (long)p.tiles_m * p.tiles_n * p.split_k * a->batch1 * a->batch2;
    if (units > 0x7fffffffL) {
        set_error("gemm_tc: too many work units");
        return LASR_ERR_UNSUPPORTED;
    }
    p.total_units = (int)units;

    p.conv_mode = 0;
    p.a_mn = a->trans_a ? 1 : 0;
    p.b_mn = a->trans_b ? 1 : 0;
    if (a->c_dtype != LASR_F32 && (p.epi_mode == EPI_RES || p.epi_mode == EPI_ACC)) p.epi_mode = EPI_GENERIC;
    CUtensorMap mc, mx;
    setup_tma_epilogue(p, &mc, &mx, a->batch1, a->batch2);
    return launch_tc(ma, mb, mc, mx, p, st);
}

// ------------------------------------------------------------------------------------------------
// Conv2d(d -> d, 3x3, stride 2) + ReLU of the sub-sampling front end (nets/subsampling.py:33-34) as an implicit GEMM.
// conv1 writes its output in PARITY PLANES  h1p[b][pt*2+pf][u*V + v][c]  (t1 = 2u+pt, f1 = 2v+pf, U x V slots per plane, pad
// slots zero), and conv2's output / output gradient live in the padded layout  y[b][t2*V + f2][c]  (V slots per t2 row,
// F2 = V-1 of them real, the rest zero in the gradient).  With the same row pitch V on both sides, tap (kh,kw) of output row
// r = t2*V+f2 reads plane (kh&1, kw&1) at row r + (kh>>1)*V + (kw>>1): every operand tile is a dense, unit-stride TMA box at a
// per-tap row offset, so the 9x im2col matrix (3.3 GB at C2/B=126) and the col2im pass never exist.
//   forward : C[b][r][co]          = relu(bias + sum_tap sum_ci h1p[b][plane][r+off][ci] W[co][tap][ci])
//   dgrad   : dh1p[b][pl][r][ci]   = relu'(h1p) * sum_{tap in class pl} sum_co dY[b][r-off][co] W[co][tap][ci]   (4 launches)
//   wgrad   : dW[co][tap][ci]     += sum_b sum_r dY[b][r][co] h1p[b][plane][r+off][ci]
// Out-of-range rows are TMA zero-fill (negative or >= extent); in-row wrap-around lands on zero slots.
// ------------------------------------------------------------------------------------------------
int conv2_tc_dispatch(int mode, int plane_class, const void* h1p, const void* w2, const float* bias, const void* dy, void* out,
                      int B, int U, int V, int T2, int d, int split_k, cudaStream_t st) {
    if (d % 64 != 0 || d > 2304 || B < 1 || U < 1 || V < 1 || T2 < 1) {
        set_error("conv2: unsupported shape d=%d", d);
        return LASR_ERR_UNSUPPORTED;
    }
    const long PR = (long)U * V;   // rows per parity plane
    const long YR = (long)T2 * V;  // rows per utterance of the padded conv2 output
    TcParams p;
    memset(&p, 0, sizeof(p));
    p.alpha = 1.f;
    p.batch2 = 1;
    p.split_k = 1;
    p.vec_ok = 1;
    p.conv_mode = mode;
    p.conv_kbt = d / BK;
    p.conv_d = d;
    int ntaps = 0;
    for (int kh = 0; kh < 3; ++kh)
        for (int kw = 0; kw < 3; ++kw) {
            const int pl = (kh & 1) * 2 + (kw & 1);
            if (mode == 2 && pl != plane_class) continue;
            p.conv_off[ntaps] = (kh >> 1) * V + (kw >> 1);
            p.conv_plane[ntaps] = pl;
            p.conv_tap[ntaps] = kh * 3 + kw;
            ++ntaps;
        }
    const int bn = d <= 256 ? d : 256;
    if (d % bn != 0) {
        set_error("conv2: d must be a multiple of the N tile");
        return LASR_ERR_UNSUPPORTED;
    }
    CUtensorMap ma, mb;
    int rc;
    if (mode == 1) {
        if ((rc = make_map(&ma, h1p, d, PR, d, 4, PR * d, B, 4 * PR * d, BK, BM))) return rc;
        if ((rc = make_map(&mb, w2, 9L * d, d, 9L * d, 1, 0, 1, 0, BK, bn))) return rc;
        p.c = out; p.bias = bias; p.c_dtype = LASR_BF16;
        p.m = (int)YR; p.n = d; p.k = 9 * d; p.n_store = d; p.ldc = d; p.sc1 = YR * d;
        p.act = LASR_ACT_RELU; p.epi_mode = EPI_RELU;
        p.a_mn = 0; p.b_mn = 0;
    } else if (mode == 2) {
        if ((rc = make_map(&ma, dy, d, YR, d, 1, 0, B, YR * d, BK, BM))) return rc;
        if ((rc = make_map(&mb, w2, 9L * d, d, 9L * d, 1, 0, 1, 0, 64, BK))) return rc;
        p.c = reinterpret_cast<bf16*>(out) + (long)plane_class * PR * d;
        p.dact = reinterpret_cast<const bf16*>(h1p) + (long)plane_class * PR * d;
        p.lddact = d; p.c_dtype = LASR_BF16;
        p.m = (int)PR; p.n = d; p.k = ntaps * d; p.n_store = d; p.ldc = d; p.sc1 = 4 * PR * d;
        p.act = LASR_ACT_RELU; p.epi_mode = EPI_DRELU;
        p.a_mn = 0; p.b_mn = 1;
    } else if (mode == 3) {
        if ((rc = make_map(&ma, dy, d, YR, d, 1, 0, B, YR * d, 64, BK))) return rc;
        if ((rc = make_map(&mb, h1p, d, PR, d, 4, PR * d, B, 4 * PR * d, 64, BK))) return rc;
        p.c = out; p.c_dtype = LASR_F32;
        p.m = d; p.n = 9 * d; p.k = (int)YR; p.n_store = 9 * d; p.ldc = 9L * d; p.sc1 = 0;
        p.accumulate = 1; p.epi_mode = EPI_ACC; p.split_k = split_k < 1 ? 1 : split_k;
        p.a_mn = 1; p.b_mn = 1;
    } else {
        set_error("conv2: bad mode");
        return LASR_ERR_BAD_ARG;
    }
    p.bn = bn;
    p.stage_bytes = A_BYTES + bn * BK * 2;
    p.stages = SM_RING_BUDGET / p.stage_bytes;
    if (p.stages > MAX_STAGES) p.stages = MAX_STAGES;
    p.tiles_m = ceil_div(p.m, BM);
    p.tiles_n = ceil_div(p.n_store, bn);
    const long units = (long)p.tiles_m * p.tiles_n * p.split_k * B;
    if (units > 0x7fffffffL) {
        set_error("conv2: too many work units");
        return LASR_ERR_UNSUPPORTED;
    }
    p.total_units = (int)units;
    CUtensorMap mc, mx;
    setup_tma_epilogue(p, &mc, &mx, B, 1);
    return launch_tc(ma, mb, mc, mx, p, st);
}

}  // namespace lasr
