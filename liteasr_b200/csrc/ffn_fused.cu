// Fused backward of a position-wise feed-forward block's two inner GEMMs (nets/feed_forward.py:18-19 backward, the block the
// encoder runs twice per Conformer layer: nets/conformer_layer.py:37-47,58-66):
//
//     dh  = alpha * (dy . W2) * g          g = act'(fc1 pre-activation), saved by the forward pass (lasr_gemm aux_deriv);
//                                          0 where the inner dropout dropped the activation
//     db1 += colsum(dh)                    fc1's bias gradient
//     dln = dh . W1                        gradient wrt the block's LayerNorm output
//
// in ONE tcgen05 kernel.  Unfused, dh (rows x f, 154 MB at C2 / B = 126) is written by the first GEMM's epilogue and read back by
// the second GEMM through HBM (102 us + 43 us per block); here a 128-row tile of dh lives only as 64-column chunks that go
// TMEM -> registers (x g) -> a shared-memory slab that is at the same time the A operand of the second MMA and the source of
// the bulk tensor store of dh (which the fc1 weight-gradient GEMM still needs).  HBM sees dy and g read once, dh and dln written
// once.
//
// Persistent, one CTA per SM, one 128-row tile at a time, f walked in chunks of 64 columns:
//   warp 0       TMA producer: W2 / W1 chunk rings (3 stages each)
//   warp 1       MMA issuer:   acc1[chunk & 1] (128 x 64 fp32, TMEM) = dy . W2[:, chunk]      (K = d; A = dy FROM TENSOR MEMORY)
//                              acc2 (128 x d fp32, TMEM)            += dh_chunk . W1[chunk, :]  (K = 64)
//                              + the bulk tensor store of every finished dh slab
//   warps 2..17  epilogue:     per tile dy rows -> TMEM (the A operand of the first MMA); per chunk acc1 -> x alpha x g -> bf16
//                              slab (+ column sums); per tile acc2 -> bf16 -> dln
// The dy tile is the A operand of 32 MMA chains per tile with only N = 64 columns each: read from shared memory it would cost
// 4 KB of operand traffic per 32-cycle instruction next to 2 KB of B -- more than the 128 B/clk a SM's shared memory delivers
// (measured: the first version of this kernel, with dy in shared memory, ran at 111 us with the L1/shared pipe 67 % busy and
// the tensor pipe 35 %).  In tensor memory it costs nothing, and the 64 KB it occupied hold a third stage of both weight rings.
// TMEM: acc1 2 x 64 columns, acc2 d <= 256 columns, dy 128 columns (two bf16 per column) = 512.  d % 64 == 0, f % 64 == 0.
#include <cuda.h>
#include <cudaTypedefs.h>

#include "common.cuh"
#include "philox.cuh"
#include "tc_ptx.cuh"

namespace lasr {
namespace ffn {

constexpr int TM = 128;   // rows per tile (MMA M)
constexpr int CN = 64;    // f columns per chunk
constexpr int EPI_W = 16;
constexpr int CTRL_W = 4;                 // warp 0 W2 loads, warp 1 MMA issue, warp 2 dh stores, warp 3 W1 loads
constexpr int THREADS = 32 * (CTRL_W + EPI_W);  // warps 4..19 epilogue
constexpr int DMAX = 256;

constexpr int W2S = 2, W1S = 3;                  // stages of the two weight rings (a W1 stage is released late: by the second MMA)
constexpr int OFF_W2 = 0;                        // W2S stages x (d/64 boxes of 64 k x 64 n, 8 KB each)
constexpr int OFF_W1 = OFF_W2 + W2S * 32768;     // W1S stages x (d/64 boxes of 64 k x 64 n)
constexpr int OFF_DH = OFF_W1 + W1S * 32768;     // 2 slabs of 128 rows x 64 bf16
constexpr int OFF_BAR = OFF_DH + 2 * 16384;
constexpr int OFF_CS = OFF_BAR + 512;            // per-CTA column sums of dh (f floats, f <= FMAX)
constexpr int FMAX = 2048;
constexpr int TM_ACC1 = 0, TM_ACC2 = 128, TM_DY = 384;  // TMEM columns
constexpr int SMEM_BYTES = OFF_CS + FMAX * 4 + 1024;
static_assert(SMEM_BYTES <= 232448, "shared-memory budget");

enum { DY_FULL = 0, DY_EMPTY, W2_FULL, W2_EMPTY = W2_FULL + W2S, W1_FULL = W2_EMPTY + W2S, W1_EMPTY = W1_FULL + W1S, ACC1_FULL = W1_EMPTY + W1S,
       ACC1_EMPTY = ACC1_FULL + 2, DH_FULL = ACC1_EMPTY + 2, DH_EMPTY = DH_FULL + 2, ACC2_FULL = DH_EMPTY + 2, ACC2_EMPTY, NBARS };

struct Params {
    const bf16* dy;  // (M, D)
    long lddy;
    const bf16* g;   // (M, F) saved activation derivative
    long ldg;
    bf16* dln;       // (M, D)
    long lddln;
    bf16* dh;        // (M, F)
    long lddh;
    float* colsum;   // (F) += column sums of dh, or nullptr
    float alpha;
    int M, D, F;
    int tiles;
    long long* trace;  // developer aid: 8 clock64 stamps per chunk of CTA 0's first tile (lasr_ffn_bwd_set_trace)
};

__device__ __forceinline__ uint4 ldg_pred_u4(const void* p, bool pred) {
    uint4 v;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %5, 0;\n\t"
        "mov.b32 %0, 0;\n\tmov.b32 %1, 0;\n\tmov.b32 %2, 0;\n\tmov.b32 %3, 0;\n\t"
        "@p ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];\n\t}"
        : "=&r"(v.x), "=&r"(v.y), "=&r"(v.z), "=&r"(v.w)
        : "l"(p), "r"((int)pred));
    return v;
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
// D[tmem] (+)= A[tmem] . B[smem]: the A operand comes from tensor memory (lane = row, one 32-bit column = two consecutive K)
__device__ __forceinline__ void tc_mma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tc_st32(uint32_t taddr, const uint32_t* r) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
          "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
          "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
          "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
// a = swish(x) and g = swish'(x) from ONE tanh (the arithmetic of gemm_tc.cu::swish_and_deriv): h = x/2, t = tanh(h)
__device__ __forceinline__ void swish_and_deriv(float x, float& a, float& g) {
    const float h = 0.5f * x;
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
    a = fmaf(h, t, h);
    g = fmaf(fmaf(h, fmaf(-t, t, 1.f), t), 0.5f, 0.5f);
}
__device__ __forceinline__ float bf_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf_hi(uint32_t u) { return __uint_as_float(u & 0xffff0000u); }

// column sums of a warp's 32 rows x 32 columns: after the five halving exchanges lane c holds the sum of column c over the 32 lanes
__device__ __forceinline__ float col_sums_32(float (&v)[32], int lane) {
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
        const bool up = (lane & s) != 0;
#pragma unroll
        for (int i = 0; i < s; ++i) {
            const float send = up ? v[i] : v[i + s];
            const float keep = up ? v[i + s] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
        }
    }
    return v[0];
}
// column sums of a warp's 32 rows x 16 columns: after the halving exchanges lane l holds the sum of column
// 8 b4 + 4 b3 + 2 b2 + b1 (b_i = bit i of l); lanes differing only in bit 0 hold the same column
__device__ __forceinline__ float col_sums_16(float (&v)[16], int lane) {
#pragma unroll
    for (int s = 16, n = 8; s >= 2; s >>= 1, n >>= 1) {
        const bool up = (lane & s) != 0;
#pragma unroll
        for (int i = 0; i < n; ++i) {
            const float send = up ? v[i] : v[i + n];
            const float keep = up ? v[i + n] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
        }
    }
    return v[0] + __shfl_xor_sync(0xffffffffu, v[0], 1);
}

// KBD = d / 64 is a template parameter: the MMA-issuing thread's loops then unroll completely and every descriptor is the
// stage's base descriptor plus an immediate.  With run-time loop bounds and a descriptor built per instruction the issuing
// thread needed ~80 cycles per tcgen05.mma (a chain of dependent integer instructions) for MMAs that execute in 32 cycles
// (N = 64): the kernel ran one chunk per 2.4 k cycles with the tensor pipe 35 % busy -- issue-bound, not data-bound.
template <int KBD>
__global__ void __launch_bounds__(THREADS, 1)
ffn_bwd_kernel(const __grid_constant__ CUtensorMap m_w2, const __grid_constant__ CUtensorMap m_w1,
               const __grid_constant__ CUtensorMap m_dh, const Params p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + OFF_BAR + 8 * NBARS);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int NC = p.F >> 6;       // chunks per tile
    // Every CTA walks the f chunks in its own rotation (chunk jj of a tile is column block (jj + rot) % NC): with a common
    // order all 148 SMs would ask the L2 for the SAME 64 KB of weights at the same moment (one line -> one slice -> 148 requests
    // in a row); rotated, the requests of a moment spread over the whole 2 MB of W1 and W2
    const int rot = (int)((blockIdx.x * 7u) % (unsigned)NC);

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&m_w2) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&m_w1) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&m_dh) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < NBARS; ++i) {
            uint32_t cnt = 1;
            if (i == ACC2_EMPTY || i == DY_FULL) cnt = EPI_W;
            if (i == ACC1_EMPTY || i == ACC1_EMPTY + 1 || i == DH_FULL || i == DH_FULL + 1) cnt = EPI_W / 2;  // one group of epilogue warps
            if (i == DH_EMPTY || i == DH_EMPTY + 1) cnt = 2;  // the second MMA has read the slab AND its bulk store has
            mbar_init(bars + i, cnt);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 4) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");

    if (warp == 0) {
        if (lane == 0) {
            // the two weight rings have producers of their own (this warp: W2, warp 3: W1): a W1 stage is released only when the
            // SECOND MMA of its chunk has completed, and a common producer walking the chunks in order would make the next W2
            // loads wait behind it (measured: one chunk per 2.4 k cycles, the first MMA waiting ~1.3 k cycles for its operand)
            uint32_t s2 = 0, ph2 = 0;
            for (int tile = blockIdx.x; tile < p.tiles; tile += gridDim.x) {
                for (int jj = 0; jj < NC; ++jj) {
                    const int j = jj + rot < NC ? jj + rot : jj + rot - NC;
                    mbar_wait(bars + W2_EMPTY + s2, ph2 ^ 1u);
                    mbar_arrive_expect_tx(bars + W2_FULL + s2, (uint32_t)(KBD * 8192));
                    for (int kb = 0; kb < KBD; ++kb)  // W2 (d, f) row-major = (K, N): box {64 n, 64 k}
                        tma_load_4d(smem + OFF_W2 + s2 * 32768 + kb * 8192, &m_w2, bars + W2_FULL + s2, j * CN, kb * 64, 0, 0);
                    if (++s2 == W2S) { s2 = 0; ph2 ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // instruction descriptors: c = f32, a = b = bf16, A K-major, B MN-major, N >> 3, M >> 4
            const uint32_t id1 = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((uint32_t)(CN >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
            const uint32_t id2 = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((uint32_t)(p.D >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
            // base descriptors (start address field = bits [0,14) in 16-byte units: adding (bytes >> 4) moves the operand)
            const uint64_t d_w2 = umma_desc(smem_u32(smem + OFF_W2), 8192, 1024), d_w1 = umma_desc(smem_u32(smem + OFF_W1), 8192, 1024),
                           d_dh = umma_desc(smem_u32(smem + OFF_DH), 16, 1024);
            uint32_t c1 = 0, c2 = 0, t = 0;
            uint32_t ws1 = 0, wp1 = 0, ws2 = 0, wp2 = 0;  // weight-ring stage / phase of the first and the second MMA
            auto mma1 = [&]() {  // acc1[c1 & 1] = dy (TMEM) . W2[:, chunk]
                const uint32_t a = c1 & 1u, aph = (c1 >> 1) & 1u;
                mbar_wait(bars + W2_FULL + ws1, wp1);
                if (p.trace && blockIdx.x == 0 && c1 < 32) p.trace[c1 * 8 + 0] = clock64();
                mbar_wait(bars + ACC1_EMPTY + a, aph ^ 1u);
                if (p.trace && blockIdx.x == 0 && c1 < 32) p.trace[c1 * 8 + 1] = clock64();
                tc_fence_after();
                const uint32_t td = tmem_base + TM_ACC1 + a * CN, ta = tmem_base + TM_DY;
                const uint64_t db = d_w2 + (uint64_t)(ws1 * (32768u >> 4));
#pragma unroll
                for (int kb = 0; kb < KBD; ++kb)
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)  // 16 K elements = 8 TMEM columns of the dy tile per instruction
                        tc_mma_bf16_ts(td, ta + kb * 32 + kk * 8, db + (uint64_t)((kb * 8192 + kk * 2048) >> 4), id1, (kb | kk) ? 1u : 0u);
                tc_commit(bars + W2_EMPTY + ws1);
                tc_commit(bars + ACC1_FULL + a);
                ++c1;
                if (++ws1 == W2S) { ws1 = 0; wp1 ^= 1u; }
            };
            for (int tile = blockIdx.x; tile < p.tiles; tile += gridDim.x, ++t) {
                const int m0 = tile * TM;
                mbar_wait(bars + DY_FULL, t & 1u);
                tc_fence_after();
                mma1();
                for (int j = 0; j < NC; ++j, ++c2) {
                    if (j + 1 < NC) mma1();
                    else tc_commit(bars + DY_EMPTY);  // every MMA reading this tile's dy has been issued
                    const uint32_t s = c2 & 1u, ph = (c2 >> 1) & 1u;
                    mbar_wait(bars + W1_FULL + ws2, wp2);
                    mbar_wait(bars + DH_FULL + s, ph);
                    if (p.trace && blockIdx.x == 0 && c2 < 32) p.trace[c2 * 8 + 2] = clock64();
                    if (j == 0) mbar_wait(bars + ACC2_EMPTY, (t & 1u) ^ 1u);
                    tc_fence_after();
                    const uint64_t da2 = d_dh + (uint64_t)(s * (16384u >> 4)), db2 = d_w1 + (uint64_t)(ws2 * (32768u >> 4));
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)  // acc2 += dh_chunk (A, K-major slab) . W1[chunk, :]
                        tc_mma_bf16(tmem_base + TM_ACC2, da2 + (uint64_t)((kk * 32) >> 4), db2 + (uint64_t)((kk * 2048) >> 4), id2, (j | kk) ? 1u : 0u);
                    tc_commit(bars + W1_EMPTY + ws2);
                    tc_commit(bars + DH_EMPTY + s);
                    if (++ws2 == W1S) { ws2 = 0; wp2 ^= 1u; }
                }
                tc_commit(bars + ACC2_FULL);
            }
        }
    } else if (warp == 3) {
        if (lane == 0) {
            uint32_t s1 = 0, ph1 = 0;
            for (int tile = blockIdx.x; tile < p.tiles; tile += gridDim.x) {
                for (int jj = 0; jj < NC; ++jj) {
                    const int j = jj + rot < NC ? jj + rot : jj + rot - NC;
                    mbar_wait(bars + W1_EMPTY + s1, ph1 ^ 1u);
                    mbar_arrive_expect_tx(bars + W1_FULL + s1, (uint32_t)(KBD * 8192));
                    for (int nb = 0; nb < KBD; ++nb)  // W1 (f, d) row-major = (K, N): box {64 n, 64 k}
                        tma_load_4d(smem + OFF_W1 + s1 * 32768 + nb * 8192, &m_w1, bars + W1_FULL + s1, nb * 64, j * CN, 0, 0);
                    if (++s1 == W1S) { s1 = 0; ph1 ^= 1u; }
                }
            }
        }
    } else if (warp == 2) {
        // dh goes to HBM straight from the MMA operand slabs, issued by a thread of its own: the slab's reuse then depends only on
        // this store and on the second MMA, not on the progress of a thread with other duties (with the stores on the MMA thread the
        // kernel ran in lockstep -- one handshake chain per chunk, 112 us; stores from registers cost 32 wavefronts each: 163 us)
        if (lane == 0) {
            uint32_t c = 0;
            for (int tile = blockIdx.x; tile < p.tiles; tile += gridDim.x) {
                const int m0 = tile * TM;
                for (int jj = 0; jj < NC; ++jj, ++c) {
                    const int j = jj + rot < NC ? jj + rot : jj + rot - NC;
                    const uint32_t s = c & 1u, ph = (c >> 1) & 1u;
                    mbar_wait(bars + DH_FULL + s, ph);
                    tma_store_4d(&m_dh, smem + OFF_DH + s * 16384, j * CN, m0, 0, 0);
                    bulk_commit();
                    bulk_wait_read<0>();
                    mbar_arrive(bars + DH_EMPTY + s);
                }
            }
        }
    } else {
        // Two groups of 8 epilogue warps take the chunks ALTERNATELY (group = chunk parity = acc1 buffer = slab): a warp's chain
        // per chunk (TMEM read -> x g -> slab -> column sums) is ~1.3 k cycles of latency, so with all 16 warps on every chunk the
        // kernel ran one chunk per chain (2.5 k cycles, tensor pipe 35 % busy); alternating groups give every chain two chunk
        // periods.  Inside a group: 2 warps per TMEM lane quarter, 32 of the chunk's 64 columns each.
        const int ew = warp - CTRL_W;
        const int q = warp & 3;             // TMEM lane quarter of this warp
        const int part = ew >> 2;           // dy / dln: 64 of the 256 columns
        const int grp = ew >> 3;            // chunk parity served by this warp
        const int half = (ew >> 2) & 1;     // 32 of a chunk's 64 columns
        const int r = q * 32 + lane;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        const float alpha = p.alpha;
        float* cs_smem = reinterpret_cast<float*>(smem + OFF_CS);
        if (p.colsum) {
            for (int i = threadIdx.x - 32 * CTRL_W; i < p.F; i += 32 * EPI_W) cs_smem[i] = 0.f;
            asm volatile("bar.sync 1, %0;" ::"n"(32 * EPI_W) : "memory");
        }
        uint32_t t = 0;
        for (int tile = blockIdx.x; tile < p.tiles; tile += gridDim.x, ++t) {
            const int row = tile * TM + r;
            const bool row_ok = row < p.M;
            const bf16* gp = p.g + (long)row * p.ldg + 32 * half;
            const int j0 = grp + rot < NC ? grp + rot : grp + rot - NC;
            uint4 gq[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) gq[i] = ldg_pred_u4(gp + j0 * CN + 8 * i, row_ok);
            {   // this warp's share of the dy tile -> tensor memory: rows 32 q .. + 31 (lanes), K elements [64 part, + 64) = 32 columns
                uint4 x[8];
                const bf16* dp = p.dy + (long)row * p.lddy + 64 * part;
#pragma unroll
                for (int i = 0; i < 8; ++i) x[i] = ldg_pred_u4(dp + 8 * i, row_ok && 64 * part + 8 * i < p.D);
                mbar_wait(bars + DY_EMPTY, (t & 1u) ^ 1u);  // every MMA that read the previous tile's dy has completed
                tc_fence_after();
                tc_st32(lane_addr + TM_DY + 32 * part, reinterpret_cast<const uint32_t*>(x));
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bars + DY_FULL);
            }
            for (int jj = grp; jj < NC; jj += 2) {
                const uint32_t c = t * (uint32_t)NC + (uint32_t)jj;  // global chunk counter (NC is even: parity of c = grp)
                const int j = jj + rot < NC ? jj + rot : jj + rot - NC;
                const uint32_t s = (uint32_t)grp, ph = (c >> 1) & 1u;
                // this group's next chunk's factors: in flight while this chunk is processed
                const bool more = jj + 2 < NC;
                const int jn = j + 2 < NC ? j + 2 : j + 2 - NC;
                uint4 nq[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) nq[i] = ldg_pred_u4(gp + jn * CN + 8 * i, row_ok && more);
                mbar_wait(bars + ACC1_FULL + s, ph);
                const bool tr = p.trace && blockIdx.x == 0 && (ew == 0 || ew == 8) && lane == 0 && c < 32;
                if (tr) p.trace[c * 8 + 3] = clock64();
                tc_fence_after();
                float v[32];
                tc_ld32(lane_addr + TM_ACC1 + s * CN + 32 * half, v);
                if (tr) p.trace[c * 8 + 4] = clock64();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bars + ACC1_EMPTY + s);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const uint32_t gw[4] = {gq[i].x, gq[i].y, gq[i].z, gq[i].w};
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        v[8 * i + 2 * e] *= alpha * bf_lo(gw[e]);
                        v[8 * i + 2 * e + 1] *= alpha * bf_hi(gw[e]);
                    }
                }
                if (tr) p.trace[c * 8 + 5] = clock64();
                mbar_wait(bars + DH_EMPTY + s, ph ^ 1u);
                if (tr) p.trace[c * 8 + 6] = clock64();
                uint8_t* rowp = smem + OFF_DH + s * 16384 + r * 128;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    uint4 u;
                    u.x = pack2(v[8 * i], v[8 * i + 1]); u.y = pack2(v[8 * i + 2], v[8 * i + 3]);
                    u.z = pack2(v[8 * i + 4], v[8 * i + 5]); u.w = pack2(v[8 * i + 6], v[8 * i + 7]);
                    *reinterpret_cast<uint4*>(rowp + (((4 * half + i) ^ (r & 7)) << 4)) = u;
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(bars + DH_FULL + s);
                if (tr) p.trace[c * 8 + 7] = clock64();
                if (p.colsum) {  // fc1's bias gradient from the fp32 values: warp tree, then one shared-memory add per column
                    const float cs = col_sums_32(v, lane);
                    atomicAdd(cs_smem + j * CN + 32 * half + lane, cs);
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) gq[i] = nq[i];
            }
            // dln tile: acc2 -> bf16 -> global (this warp: its 32 rows x 64 columns)
            mbar_wait(bars + ACC2_FULL, t & 1u);
            tc_fence_after();
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int cc = part * 64 + i * 16;
                if (cc < p.D) {  // warp-uniform
                    float v[16];
                    tc_ld16(lane_addr + TM_ACC2 + cc, v);
                    if (row_ok) {
                        uint4* dst = reinterpret_cast<uint4*>(p.dln + (long)row * p.lddln + cc);
                        uint4 u;
                        u.x = pack2(v[0], v[1]); u.y = pack2(v[2], v[3]); u.z = pack2(v[4], v[5]); u.w = pack2(v[6], v[7]);
                        dst[0] = u;
                        u.x = pack2(v[8], v[9]); u.y = pack2(v[10], v[11]); u.z = pack2(v[12], v[13]); u.w = pack2(v[14], v[15]);
                        dst[1] = u;
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bars + ACC2_EMPTY);
        }
        if (p.colsum) {  // the CTA's column sums: one global add per column per CTA
            asm volatile("bar.sync 1, %0;" ::"n"(32 * EPI_W) : "memory");
            for (int i = threadIdx.x - 32 * CTRL_W; i < p.F; i += 32 * EPI_W) atomicAdd(p.colsum + i, cs_smem[i]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// =================================================================================================================================
// Fused FORWARD of the same block (nets/feed_forward.py:18-19 inside nets/conformer_layer.py:37-47,58-66):
//
//     h   = ln . W1^T + b1                               (never stored)
//     a   = drop_in(swish(h))            -> HBM (bf16)   fc2's weight gradient needs it
//     g   = swish'(h), 0 where dropped   -> HBM (bf16)   what the fused backward above multiplies by
//     out = res + drop_out(alpha * (a . W2^T + b2))      -> HBM (fp32 residual stream)
//
// STATUS: correct (a and g bit-identical to the GEMM pair, tests/test_ffn_fused_gpu.py) but NOT faster, so engine.py keeps it behind
// LASR_FUSED_FFN_FWD=1: 137 us per block against 75 + 51 us for lasr_gemm(Swish, aux_deriv) + lasr_gemm(res) without dropout, 153
// against 91 + 53 us with the shipped rates (tools/ffn_bench.py ... fwd0.1).  fc1 is bound by its epilogue's instruction stream
// (~500 instructions per thread and 32-column chunk: bias, tanh, the Swish / Swish' FMAs, packs, staging stores; Philox on top), and
// this kernel executes the same epilogue with 8 of its 16 epilogue warps per chunk plus the second contraction's handshakes -- one
// 64-column chunk per ~4 k cycles -- which costs more than the 154 MB read of a that it saves (profiles/r2_ffn_fwd.txt).
// Unfused, a (154 MB at C2 / B = 126) is written by fc1's epilogue and read back by fc2; here a 128-row tile of a exists as 64-column chunks that go
// TMEM -> registers (bias, one tanh for swish and swish', Philox masks) -> a shared-memory slab that is at the same time the A
// operand of the second MMA and the source of the bulk tensor store; the second contraction rides under the first one's epilogue.
// Same skeleton as the backward kernel: ln tile = A operand of the first MMA from TENSOR MEMORY, two alternating groups of 8
// epilogue warps, separate producers for the two weight rings, a store thread.
//   warp 0: W1 chunk loads (2 stages)   warp 1: MMA issue   warp 2: bulk stores of the a / g slabs   warp 3: W2 chunk loads (3 stages)
// TMEM: acc1 2 x 64 columns, acc2 d columns, ln 128 columns.
// =================================================================================================================================
constexpr int F_R1S = 2, F_R2S = 3;
constexpr int FOFF_R1 = 0;                            // W1 chunk ring: d/64 boxes of {64 k, 64 n} (K-major B of the first MMA)
constexpr int FOFF_R2 = FOFF_R1 + F_R1S * 32768;      // W2 chunk ring: one box {64 k, d n}        (K-major B of the second MMA)
constexpr int FOFF_A = FOFF_R2 + F_R2S * 32768;       // 2 a slabs of 128 rows x 64 bf16 (K-major A of the second MMA)
constexpr int FOFF_G = FOFF_A + 2 * 16384;            // 2 g slabs (store staging only)
constexpr int FOFF_BAR = FOFF_G + 2 * 16384;
constexpr int FSMEM_BYTES = FOFF_BAR + 512 + 1024;
static_assert(FSMEM_BYTES <= 232448, "shared-memory budget (forward)");

enum { F_LN_FULL = 0, F_LN_EMPTY, F_R1_FULL, F_R1_EMPTY = F_R1_FULL + F_R1S, F_R2_FULL = F_R1_EMPTY + F_R1S, F_R2_EMPTY = F_R2_FULL + F_R2S,
       F_ACC1_FULL = F_R2_EMPTY + F_R2S, F_ACC1_EMPTY = F_ACC1_FULL + 2, F_SLAB_FULL = F_ACC1_EMPTY + 2, F_SLAB_EMPTY = F_SLAB_FULL + 2,
       F_ACC2_FULL = F_SLAB_EMPTY + 2, F_ACC2_EMPTY, F_NBARS };

struct FwdParams {
    const bf16* ln;    // (M, D)
    long ldln;
    const float* b1;   // (F)
    const float* b2;   // (D)
    const float* res;  // (M, D) fp32
    long ldres;
    float* out;        // (M, D) fp32
    long ldout;
    float alpha;       // block scale (0.5 for the macaron halves)
    int M, D, F, tiles;
    DropCfg drop_in, drop_out;
};

template <int KBD>
__global__ void __launch_bounds__(THREADS, 1)
ffn_fwd_kernel(const __grid_constant__ CUtensorMap m_w1, const __grid_constant__ CUtensorMap m_w2, const __grid_constant__ CUtensorMap m_a,
               const __grid_constant__ CUtensorMap m_g, const FwdParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + FOFF_BAR);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + FOFF_BAR + 8 * F_NBARS);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int NC = p.F >> 6;
    const int rot = (int)((blockIdx.x * 7u) % (unsigned)NC);  // per-CTA chunk rotation (see the backward kernel)

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&m_w1) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&m_w2) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&m_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&m_g) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < F_NBARS; ++i) {
            uint32_t cnt = 1;
            if (i == F_ACC2_EMPTY || i == F_LN_FULL) cnt = EPI_W;
            if (i == F_ACC1_EMPTY || i == F_ACC1_EMPTY + 1 || i == F_SLAB_FULL || i == F_SLAB_FULL + 1) cnt = EPI_W / 2;
            if (i == F_SLAB_EMPTY || i == F_SLAB_EMPTY + 1) cnt = 2;  // the second MMA has read the a slab AND both bulk stores have
            mbar_init(bars + i, cnt);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 4) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");

    if (warp == 0) {
        if (lane == 0) {
            uint32_t s1 = 0, ph1 = 0;
            for (int tile = blockIdx.x; tile < p.tiles; tile += gridDim.x) {
                for (int jj = 0; jj < NC; ++jj) {
                    const int j = jj + rot < NC ? jj + rot : jj + rot - NC;
                    mbar_wait(bars + F_R1_EMPTY + s1, ph1 ^ 1u);
                    mbar_arrive_expect_tx(bars + F_R1_FULL + s1, (uint32_t)(KBD * 8192));
                    for (int kb = 0; kb < KBD; ++kb)  // W1 (f, d) row-major = (N, K): box {64 k, 64 n}
                        tma_load_4d(smem + FOFF_R1 + s1 * 32768 + kb * 8192, &m_w1, bars + F_R1_FULL + s1, kb * 64, j * CN, 0, 0);
                    if (++s1 == F_R1S) { s1 = 0; ph1 ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // c = f32, a = b = bf16, both operands K-major, N >> 3, M >> 4
            const uint32_t id1 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(CN >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
            const uint32_t id2 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.D >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
            const uint64_t d_r1 = umma_desc(smem_u32(smem + FOFF_R1), 16, 1024), d_r2 = umma_desc(smem_u32(smem + FOFF_R2), 16, 1024),
                           d_a = umma_desc(smem_u32(smem + FOFF_A), 16, 1024);
            uint32_t c1 = 0, c2 = 0, t = 0;
            uint32_t ws1 = 0, wp1 = 0, ws2 = 0, wp2 = 0;
            auto mma1 = [&]() {  // acc1[c1 & 1] = ln (TMEM) . W1[chunk, :]^T
                const uint32_t a = c1 & 1u, aph = (c1 >> 1) & 1u;
                mbar_wait(bars + F_R1_FULL + ws1, wp1);
                mbar_wait(bars + F_ACC1_EMPTY + a, aph ^ 1u);
                tc_fence_after();
                const uint32_t td = tmem_base + TM_ACC1 + a * CN, ta = tmem_base + TM_DY;
                const uint64_t db = d_r1 + (uint64_t)(ws1 * (32768u >> 4));
#pragma unroll
                for (int kb = 0; kb < KBD; ++kb)
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)
                        tc_mma_bf16_ts(td, ta + kb * 32 + kk * 8, db + (uint64_t)((kb * 8192 + kk * 32) >> 4), id1, (kb | kk) ? 1u : 0u);
                tc_commit(bars + F_R1_EMPTY + ws1);
                tc_commit(bars + F_ACC1_FULL + a);
                ++c1;
                if (++ws1 == F_R1S) { ws1 = 0; wp1 ^= 1u; }
            };
            for (int tile = blockIdx.x; tile < p.tiles; tile += gridDim.x, ++t) {
                mbar_wait(bars + F_LN_FULL, t & 1u);
                tc_fence_after();
                mma1();
                for (int j = 0; j < NC; ++j, ++c2) {
                    if (j + 1 < NC) mma1();
                    else tc_commit(bars + F_LN_EMPTY);  // every MMA reading this tile's ln has been issued
                    const uint32_t s = c2 & 1u, ph = (c2 >> 1) & 1u;
                    mbar_wait(bars + F_R2_FULL + ws2, wp2);
                    mbar_wait(bars + F_SLAB_FULL + s, ph);
                    if (j == 0) mbar_wait(bars + F_ACC2_EMPTY, (t & 1u) ^ 1u);
                    tc_fence_after();
                    const uint64_t da2 = d_a + (uint64_t)(s * (16384u >> 4)), db2 = d_r2 + (uint64_t)(ws2 * (32768u >> 4));
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)  // acc2 += a_chunk (K-major slab) . W2[:, chunk]^T
                        tc_mma_bf16(tmem_base + TM_ACC2, da2 + (uint64_t)((kk * 32) >> 4), db2 + (uint64_t)((kk * 32) >> 4), id2, (j | kk) ? 1u : 0u);
                    tc_commit(bars + F_R2_EMPTY + ws2);
                    tc_commit(bars + F_SLAB_EMPTY + s);
                    if (++ws2 == F_R2S) { ws2 = 0; wp2 ^= 1u; }
                }
                tc_commit(bars + F_ACC2_FULL);
            }
        }
    } else if (warp == 3) {
        if (lane == 0) {
            uint32_t s2 = 0, ph2 = 0;
            for (int tile = blockIdx.x; tile < p.tiles; tile += gridDim.x) {
                for (int jj = 0; jj < NC; ++jj) {
                    const int j = jj + rot < NC ? jj + rot : jj + rot - NC;
                    mbar_wait(bars + F_R2_EMPTY + s2, ph2 ^ 1u);
                    mbar_arrive_expect_tx(bars + F_R2_FULL + s2, (uint32_t)(p.D * 128));
                    tma_load_4d(smem + FOFF_R2 + s2 * 32768, &m_w2, bars + F_R2_FULL + s2, j * CN, 0, 0, 0);  // W2 (d, f): box {64 k, d n}
                    if (++s2 == F_R2S) { s2 = 0; ph2 ^= 1u; }
                }
            }
        }
    } else if (warp == 2) {
        if (lane == 0) {
            uint32_t c = 0;
            for (int tile = blockIdx.x; tile < p.tiles; tile += gridDim.x) {
                const int m0 = tile * TM;
                for (int jj = 0; jj < NC; ++jj, ++c) {
                    const int j = jj + rot < NC ? jj + rot : jj + rot - NC;
                    const uint32_t s = c & 1u, ph = (c >> 1) & 1u;
                    mbar_wait(bars + F_SLAB_FULL + s, ph);
                    tma_store_4d(&m_a, smem + FOFF_A + s * 16384, j * CN, m0, 0, 0);
                    tma_store_4d(&m_g, smem + FOFF_G + s * 16384, j * CN, m0, 0, 0);
                    bulk_commit();
                    bulk_wait_read<0>();
                    mbar_arrive(bars + F_SLAB_EMPTY + s);
                }
            }
        }
    } else {
        const int ew = warp - CTRL_W;
        const int q = warp & 3;             // TMEM lane quarter of this warp
        const int part = ew >> 2;           // ln / out: 64 of the 256 columns
        const int grp = ew >> 3;            // chunk parity served by this warp
        const int half = (ew >> 2) & 1;     // 32 of a chunk's 64 columns
        const int r = q * 32 + lane;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        const bool din = p.drop_in.thr != 0, dout = p.drop_out.thr != 0;  // uniform
        DropKey dki = {}, dko = {};
        if (din) dki = drop_key(p.drop_in);
        if (dout) dko = drop_key(p.drop_out);
        const float sc_in = din ? dki.scale : 1.f;
        const float alpha_s = dout ? p.alpha * dko.scale : p.alpha;
        uint32_t t = 0;
        for (int tile = blockIdx.x; tile < p.tiles; tile += gridDim.x, ++t) {
            const int row = tile * TM + r;
            const bool row_ok = row < p.M;
            {   // this warp's share of the ln tile -> tensor memory
                uint4 x[8];
                const bf16* dp = p.ln + (long)row * p.ldln + 64 * part;
#pragma unroll
                for (int i = 0; i < 8; ++i) x[i] = ldg_pred_u4(dp + 8 * i, row_ok && 64 * part + 8 * i < p.D);
                mbar_wait(bars + F_LN_EMPTY, (t & 1u) ^ 1u);
                tc_fence_after();
                tc_st32(lane_addr + TM_DY + 32 * part, reinterpret_cast<const uint32_t*>(x));
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bars + F_LN_FULL);
            }
            for (int jj = grp; jj < NC; jj += 2) {
                const uint32_t c = t * (uint32_t)NC + (uint32_t)jj;
                const int j = jj + rot < NC ? jj + rot : jj + rot - NC;
                const uint32_t s = (uint32_t)grp, ph = (c >> 1) & 1u;
                const int col0 = j * CN + 32 * half;
                mbar_wait(bars + F_ACC1_FULL + s, ph);
                tc_fence_after();
                float v[32];
                tc_ld32_issue(lane_addr + TM_ACC1 + s * CN + 32 * half, v);
                uint32_t mk[16];  // packed keep masks of this thread's 32 columns, evaluated while the TMEM load is in flight
                if (din) {
                    uint32_t h0[8], h1[8];
                    drop_masks16(dki, (uint32_t)row, (uint32_t)col0 >> 4, h0);
                    drop_masks16(dki, (uint32_t)row, ((uint32_t)col0 >> 4) + 1u, h1);
#pragma unroll
                    for (int i = 0; i < 8; ++i) { mk[i] = h0[i]; mk[8 + i] = h1[i]; }
                }
                tc_ld_wait32(v);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bars + F_ACC1_EMPTY + s);
                // (finishing all 32 columns in registers BEFORE this wait measured slower: 148 vs 137 us per block)
                mbar_wait(bars + F_SLAB_EMPTY + s, ph ^ 1u);
                uint8_t* arow = smem + FOFF_A + s * 16384 + r * 128;
                uint8_t* grow = smem + FOFF_G + s * 16384 + r * 128;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float4 ba = __ldg(reinterpret_cast<const float4*>(p.b1 + col0 + 8 * i));
                    const float4 bb = __ldg(reinterpret_cast<const float4*>(p.b1 + col0 + 8 * i + 4));
                    const float bv[8] = {ba.x, ba.y, ba.z, ba.w, bb.x, bb.y, bb.z, bb.w};
                    float a[8], g[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        swish_and_deriv(v[8 * i + e] + bv[e], a[e], g[e]);
                        a[e] *= sc_in;
                    }
                    uint4 ua, ug;
                    ua.x = pack2(a[0], a[1]); ua.y = pack2(a[2], a[3]); ua.z = pack2(a[4], a[5]); ua.w = pack2(a[6], a[7]);
                    ug.x = pack2(g[0], g[1]); ug.y = pack2(g[2], g[3]); ug.z = pack2(g[4], g[5]); ug.w = pack2(g[6], g[7]);
                    if (din) {
                        ua.x &= mk[4 * i]; ua.y &= mk[4 * i + 1]; ua.z &= mk[4 * i + 2]; ua.w &= mk[4 * i + 3];
                        ug.x &= mk[4 * i]; ug.y &= mk[4 * i + 1]; ug.z &= mk[4 * i + 2]; ug.w &= mk[4 * i + 3];
                    }
                    const int off = ((4 * half + i) ^ (r & 7)) << 4;
                    *reinterpret_cast<uint4*>(arow + off) = ua;
                    *reinterpret_cast<uint4*>(grow + off) = ug;
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(bars + F_SLAB_FULL + s);
            }
            // out tile: res + keep * scale * alpha * (acc2 + b2) -> fp32 (this warp: its 32 rows x 64 columns)
            mbar_wait(bars + F_ACC2_FULL, t & 1u);
            tc_fence_after();
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int cc = part * 64 + i * 16;
                if (cc < p.D) {  // warp-uniform
                    float4 rr[4];
                    const float* rp = p.res + (long)row * p.ldres + cc;
#pragma unroll
                    for (int e = 0; e < 4; ++e) rr[e] = ldg_pred_f4(rp + 4 * e, row_ok);
                    uint32_t keep = 0xffffu;
                    if (dout) keep = drop_keep16(dko, (uint32_t)row, (uint32_t)cc >> 4);
                    float v[16];
                    tc_ld16(lane_addr + TM_ACC2 + cc, v);
                    if (row_ok) {
                        float4* dst = reinterpret_cast<float4*>(p.out + (long)row * p.ldout + cc);
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const float4 b = __ldg(reinterpret_cast<const float4*>(p.b2 + cc + 4 * e));
                            float4 o;
                            o.x = fmaf(v[4 * e], alpha_s, alpha_s * b.x); o.y = fmaf(v[4 * e + 1], alpha_s, alpha_s * b.y);
                            o.z = fmaf(v[4 * e + 2], alpha_s, alpha_s * b.z); o.w = fmaf(v[4 * e + 3], alpha_s, alpha_s * b.w);
                            const uint32_t k4 = keep >> (4 * e);
                            o.x = ((k4 & 1u) ? o.x : 0.f) + rr[e].x; o.y = ((k4 & 2u) ? o.y : 0.f) + rr[e].y;
                            o.z = ((k4 & 4u) ? o.z : 0.f) + rr[e].z; o.w = ((k4 & 8u) ? o.w : 0.f) + rr[e].w;
                            dst[e] = o;
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bars + F_ACC2_EMPTY);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}


static PFN_cuTensorMapEncodeTiled_v12000 encoder() {
    static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
    if (!fn) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(ptr);
    }
    return fn;
}

// bf16 matrix (rows, inner) with row stride ld; box {64 inner, box_rows}, SWIZZLE_128B
static int make_map(CUtensorMap* map, const void* base, long inner, long rows, long ld, int box_rows, bool store) {
    auto enc = encoder();
    if (!enc) { set_error("cuTensorMapEncodeTiled entry point unavailable"); return LASR_ERR_DRIVER; }
    const cuuint64_t row_bytes = (cuuint64_t)ld * 2;
    cuuint64_t dims[4] = {(cuuint64_t)inner, (cuuint64_t)rows, 1, 1};
    cuuint64_t strides[3] = {row_bytes, row_bytes, row_bytes};
    cuuint32_t box[4] = {64, (cuuint32_t)box_rows, 1, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (row_bytes & 15)) {
        set_error("ffn_bwd: operand base / row stride must be 16-byte aligned (base=%p ld=%ld)", base, ld);
        return LASR_ERR_BAD_ARG;
    }
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                     store ? CU_TENSOR_MAP_L2_PROMOTION_NONE : CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("ffn_bwd: cuTensorMapEncodeTiled failed (%d): inner=%ld rows=%ld ld=%ld", (int)r, inner, rows, ld);
        return LASR_ERR_DRIVER;
    }
    return LASR_OK;
}

}  // namespace ffn
}  // namespace lasr

extern "C" {
using namespace lasr;

static long long* g_ffn_trace = nullptr;
/* developer aid: device buffer of 32 x 8 int64 receiving clock64 stamps of CTA 0's first 32 chunks (NULL = off) */
void lasr_ffn_bwd_set_trace(void* buf) { g_ffn_trace = reinterpret_cast<long long*>(buf); }

int lasr_ffn_bwd_supported(int d, int f) { return (d >= 64 && d <= ffn::DMAX && d % 64 == 0 && f >= 128 && f % 128 == 0 && f <= ffn::FMAX) ? 1 : 0; }

int lasr_ffn_bwd(const void* dy, int64_t lddy, const void* g, int64_t ldg, const void* w2, int64_t ldw2, const void* w1, int64_t ldw1,
                 void* dh, int64_t lddh, void* dln, int64_t lddln, float* colsum, float alpha, int M, int d, int f, void* stream) {
    LASR_REQUIRE(dy && g && w2 && w1 && dh && dln && M > 0, "ffn_bwd: null operand or empty problem");
    if (!lasr_ffn_bwd_supported(d, f)) {
        set_error("ffn_bwd: needs d %% 64 == 0, 64 <= d <= %d, f %% 128 == 0, f <= %d (got d=%d f=%d)", ffn::DMAX, ffn::FMAX, d, f);
        return LASR_ERR_UNSUPPORTED;
    }
    LASR_REQUIRE(lddh % 8 == 0 && (reinterpret_cast<uintptr_t>(dh) & 15) == 0, "ffn_bwd: dh must be 16-byte aligned with a row stride that is a multiple of 8");
    LASR_REQUIRE(ldg % 8 == 0 && lddln % 8 == 0 && (reinterpret_cast<uintptr_t>(g) & 15) == 0 && (reinterpret_cast<uintptr_t>(dln) & 15) == 0,
                 "ffn_bwd: g and dln must be 16-byte aligned with row strides that are multiples of 8");
    LASR_REQUIRE(lddy % 8 == 0 && (reinterpret_cast<uintptr_t>(dy) & 15) == 0, "ffn_bwd: dy must be 16-byte aligned with a row stride that is a multiple of 8");
    CUtensorMap m_w2, m_w1, m_dh;
    int rc;
    if ((rc = ffn::make_map(&m_w2, w2, f, d, ldw2, 64, false)) != LASR_OK) return rc;   // (d, f): inner = f (N), rows = d (K)
    if ((rc = ffn::make_map(&m_w1, w1, d, f, ldw1, 64, false)) != LASR_OK) return rc;   // (f, d): inner = d (N), rows = f (K)
    if ((rc = ffn::make_map(&m_dh, dh, f, M, lddh, ffn::TM, true)) != LASR_OK) return rc;
    typedef void (*Kern)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const ffn::Params);
    Kern kern = d == 256 ? ffn::ffn_bwd_kernel<4> : d == 192 ? ffn::ffn_bwd_kernel<3> : d == 128 ? ffn::ffn_bwd_kernel<2> : ffn::ffn_bwd_kernel<1>;
    static bool configured[5] = {false, false, false, false, false};
    if (!configured[d >> 6]) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, ffn::SMEM_BYTES) != cudaSuccess)
            return check_launch("ffn_bwd smem attr");
        configured[d >> 6] = true;
    }
    ffn::Params p;
    p.dy = reinterpret_cast<const bf16*>(dy); p.lddy = lddy;
    p.g = reinterpret_cast<const bf16*>(g); p.ldg = ldg;
    p.dln = reinterpret_cast<bf16*>(dln); p.lddln = lddln;
    p.dh = reinterpret_cast<bf16*>(dh); p.lddh = lddh;
    p.colsum = colsum; p.alpha = alpha;
    p.M = M; p.D = d; p.F = f;
    p.tiles = (M + ffn::TM - 1) / ffn::TM;
    p.trace = g_ffn_trace;
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
    }
    const int grid = p.tiles < sms ? p.tiles : sms;
    launch_pdl(kern, dim3((unsigned)grid), dim3(ffn::THREADS), (size_t)ffn::SMEM_BYTES, (cudaStream_t)stream, m_w2, m_w1, m_dh, p);
    return check_launch("ffn_bwd");
}

int lasr_ffn_fwd_supported(int d, int f) { return lasr_ffn_bwd_supported(d, f); }

int lasr_ffn_fwd(const void* ln, int64_t ldln, const void* w1, int64_t ldw1, const float* b1, const void* w2, int64_t ldw2, const float* b2,
                 const float* res, int64_t ldres, void* a, int64_t lda, void* g, int64_t ldg, float* out, int64_t ldout, float alpha, int M, int d,
                 int f, const void* drop_state, uint32_t in_site, uint32_t in_thr, float in_scale, uint32_t out_site, uint32_t out_thr,
                 float out_scale, void* stream) {
    LASR_REQUIRE(ln && w1 && b1 && w2 && b2 && res && a && g && out && M > 0, "ffn_fwd: null operand or empty problem");
    if (!lasr_ffn_fwd_supported(d, f)) {
        set_error("ffn_fwd: needs d %% 64 == 0, 64 <= d <= %d, f %% 128 == 0, f <= %d (got d=%d f=%d)", ffn::DMAX, ffn::FMAX, d, f);
        return LASR_ERR_UNSUPPORTED;
    }
    LASR_REQUIRE(ldln % 8 == 0 && (reinterpret_cast<uintptr_t>(ln) & 15) == 0, "ffn_fwd: ln must be 16-byte aligned with a row stride that is a multiple of 8");
    LASR_REQUIRE(ldres % 4 == 0 && ldout % 4 == 0 && ((reinterpret_cast<uintptr_t>(res) | reinterpret_cast<uintptr_t>(out)) & 15) == 0,
                 "ffn_fwd: res / out must be 16-byte aligned with row strides that are multiples of 4");
    LASR_REQUIRE(((reinterpret_cast<uintptr_t>(b1) | reinterpret_cast<uintptr_t>(b2)) & 15) == 0, "ffn_fwd: biases must be 16-byte aligned");
    LASR_REQUIRE((in_thr == 0 && out_thr == 0) || drop_state, "ffn_fwd: dropout needs drop_state");
    LASR_REQUIRE(in_thr <= LASR_DROP_THR_MAX && out_thr <= LASR_DROP_THR_MAX, "ffn_fwd: thr = round(p * 32768) <= 0x7c00");
    CUtensorMap m_w1, m_w2, m_a, m_g;
    int rc;
    if ((rc = ffn::make_map(&m_w1, w1, d, f, ldw1, 64, false)) != LASR_OK) return rc;   // (f, d): inner = d (K), rows = f (N)
    if ((rc = ffn::make_map(&m_w2, w2, f, d, ldw2, d, false)) != LASR_OK) return rc;    // (d, f): inner = f (K), rows = d (N), box {64, d}
    if ((rc = ffn::make_map(&m_a, a, f, M, lda, ffn::TM, true)) != LASR_OK) return rc;
    if ((rc = ffn::make_map(&m_g, g, f, M, ldg, ffn::TM, true)) != LASR_OK) return rc;
    typedef void (*Kern)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const ffn::FwdParams);
    Kern kern = d == 256 ? ffn::ffn_fwd_kernel<4> : d == 192 ? ffn::ffn_fwd_kernel<3> : d == 128 ? ffn::ffn_fwd_kernel<2> : ffn::ffn_fwd_kernel<1>;
    static bool configured[5] = {false, false, false, false, false};
    if (!configured[d >> 6]) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, ffn::FSMEM_BYTES) != cudaSuccess)
            return check_launch("ffn_fwd smem attr");
        configured[d >> 6] = true;
    }
    ffn::FwdParams p;
    p.ln = reinterpret_cast<const bf16*>(ln); p.ldln = ldln;
    p.b1 = b1; p.b2 = b2;
    p.res = res; p.ldres = ldres;
    p.out = out; p.ldout = ldout;
    p.alpha = alpha;
    p.M = M; p.D = d; p.F = f;
    p.tiles = (M + ffn::TM - 1) / ffn::TM;
    p.drop_in.state = p.drop_out.state = reinterpret_cast<const unsigned long long*>(drop_state);
    p.drop_in.site = in_site; p.drop_in.thr = in_thr; p.drop_in.scale = in_scale;
    p.drop_out.site = out_site; p.drop_out.thr = out_thr; p.drop_out.scale = out_scale;
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
    }
    const int grid = p.tiles < sms ? p.tiles : sms;
    launch_pdl(kern, dim3((unsigned)grid), dim3(ffn::THREADS), (size_t)ffn::FSMEM_BYTES, (cudaStream_t)stream, m_w1, m_w2, m_a, m_g, p);
    return check_launch("ffn_fwd");
}

}  // extern "C"
