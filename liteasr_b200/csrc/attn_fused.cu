// Fused relative-position self-attention forward for one Conformer layer (nets/attention.py:99-154 of the reference):
//
//   ac = (q + u) . K^T          bd = (q + v) . P^T          s = (ac + rel_shift(bd)) / sqrt(dk)
//   s[j >= klen] = -1e38        p = softmax_j(s)            O = p . V
//
// in ONE kernel per layer: both score contractions and p.V run on tcgen05 with TMEM accumulators, the legacy rel_shift,
// scale, key-padding mask and softmax happen between them on chip, and the only HBM traffic is the operands (q+u, q+v, K, P,
// V: 2 B per element, L2-resident across the tiles of a head), the bf16 probabilities the backward pass needs (written once
// by bulk tensor stores straight from the shared-memory tile that also feeds the p.V MMA) and O.  The unfused path
// (two GEMMs -> fp32 score tensors -> attn_softmax_fwd -> GEMM) moves ~10x the bytes.
//
// One CTA per (batch, head, row tile); T <= 320 keys, dk = 64.
//
// The legacy rel_shift (quirk Q1) is a flat re-view: pad a zero column in front of bd (T x (T+1)), view the same memory as
// (T+1) x T and drop the first row, i.e. out[i][j] = flat[(i+1) T + j] with flat[r (T+1)] = 0 and flat[r (T+1) + 1 + c] =
// bd[r][c].  So the tile's bd rows are written CONTIGUOUSLY into a flat shared-memory buffer at r (T+1) + 1 + c and the
// shifted rows are read back CONTIGUOUSLY at r T + j -- no per-element index arithmetic.  Output row i needs bd rows i and
// i + 1, hence a 128-row MMA tile yields 127 attention rows (tile stride 127).
//
//   thread 0    between its own worker phases: TMA ((q+v) tile + P, (q+u) tile + K, V into P's buffer once the bd MMAs
//               retired, at the end the bulk tensor stores of the probability tile) and MMA issue
//               (bd -> TMEM[0,320) ; (drained) ac -> TMEM[0,320) ; p.V -> TMEM[320,384)) -- the two roles are sequential
//   16 warps    four per TMEM lane quarter, each owning 80 of the 320 columns of its 32 rows, held in registers
//               (16 warps = 128 registers per thread; the phases are latency chains per warp, so the warp count hides them):
//               shift : bd row (TMEM) -> * scale*log2(e) -> fp16 -> flat buffer
//               pass A: s = ac * scale*log2(e) + shifted bd, mask; the 80 values stay in registers
//               pass B: e = 2^(s - m) against the warp's own row maximum m, partial sum; ONE exchange of (m, sum) per row
//               pass C: p = e * 2^(m - max) / total -> bf16 -> the K-major SWIZZLE_128B tile (aliases the flat buffer: all
//                       its reads happened in pass A) that is both the A operand of p.V and the source of the stores
//               O     : TMEM[320,384) -> bf16 -> global
#include <cuda_fp16.h>

#include <cstring>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace lasr {
namespace fa {

constexpr int TM = 128;      // bd rows per tile (MMA M)
constexpr int TOUT = 127;    // attention rows per tile
constexpr int TKMAX = 320;   // keys
constexpr int NHALF = 160;   // MMA N of one score half
constexpr int DK = 64;
constexpr int EPI_W = 16;     // four warps per TMEM lane quarter, each owning 80 of the 320 columns of its 32 rows
constexpr int PARTW = TKMAX / 4;
constexpr int CH = 16;        // columns per TMEM load / store
constexpr int THREADS = 32 * EPI_W;

// Flat fp16 shift buffer: position L = r (T+1) + c + (r0 + 1 - T) of bd[r0 + r][c] ranges over [1 - T, 128 T + 127], so with
// FLAT_PAD elements in front no write needs a bounds check.  The 5 x (128 x 64) bf16 probability slabs alias its start.
constexpr int FLAT_PAD = TKMAX;
constexpr int OFF_STG = 0;
constexpr int STG_BYTES = ((FLAT_PAD + 129 * TKMAX + 128) * 2 + 1023) / 1024 * 1024;  // 83968 (>= 5 * 128 * 128 = 81920)
constexpr int OFF_QU = OFF_STG + STG_BYTES;       // (q+u) tile, 128 x 64 bf16
constexpr int OFF_QV = OFF_QU + TM * 128;         // (q+v) tile
constexpr int OFF_K = OFF_QV + TM * 128;          // K: two 160-row halves
constexpr int OFF_P = OFF_K + 2 * NHALF * 128;    // P: two 160-row halves; later V: five 64-key atoms
constexpr int OFF_BAR = OFF_P + 2 * NHALF * 128;
constexpr int OFF_RED = OFF_BAR + 128;            // [max | sum][column part][row]
constexpr int SMEM_BYTES = OFF_RED + 2 * 4 * TM * 4 + 1024;
static_assert(STG_BYTES >= 5 * TM * 128 && SMEM_BYTES <= 232448, "shared-memory budget");

enum { BAR_BDIN = 0, BAR_ACIN, BAR_V, BAR_BD_DONE, BAR_BD_DRAINED, BAR_AC_DONE, BAR_S_DRAINED, BAR_P_READY, BAR_O_DONE, BAR_O_DRAINED, NBARS };

struct Params {
    bf16* o;
    long ldo;
    const int64_t* lens;
    int mask_mode;
    float c2;  // scale * log2(e)
    int B, H, T, ld, tiles;
    long long* trace;  // developer aid (lasr_rel_attn_fwd_set_trace): 16 clock64 stamps per CTA from one epilogue warp
};

#define FA_STAMP(i)                                                                  \
    do {                                                                             \
        if (p.trace && warp == 6 && lane == 0) p.trace[(long)tt * 16 + (i)] = clock64(); \
    } while (0)

__device__ __forceinline__ void tc_st32(uint32_t taddr, const float* v) {
    const uint32_t* r = reinterpret_cast<const uint32_t*>(v);
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
          "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
          "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
          "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
__device__ __forceinline__ void tc_st16(uint32_t taddr, const float* v) {
    const uint32_t* r = reinterpret_cast<const uint32_t*>(v);
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
          "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
// two fp32 -> packed fp16 (lo = a, hi = b), round to nearest, saturating to +-65504 (F2FP.SATFINITE.F16.F32.PACK_AB)
__device__ __forceinline__ uint32_t f16x2_sat(float a, float b) {
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
}
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void epi_barrier() { asm volatile("bar.sync 1, %0;" ::"n"(32 * EPI_W) : "memory"); }
__device__ __forceinline__ float ex2_fast(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}

// 16 x 16 columns of one TMEM row: all loads in flight before the single wait (the phases are latency chains per warp)
__device__ __forceinline__ void tc_ld16_issue(uint32_t taddr, float* v) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Control-thread steps, out of line: their descriptors and coordinates must not occupy registers of the 512 worker threads
// (the workers hold 80 score columns each).
struct Ctl {
    uint8_t* smem;
    uint64_t* bars;
    uint32_t tmem_base;
    int H, tiles, T, ld;
};
__device__ __noinline__ void ctl_bd_loads(const Ctl& c, const CUtensorMap* m_qv, const CUtensorMap* m_p, int tt) {
    const int tile = tt % c.tiles, bh = tt / c.tiles;
    const int h = bh % c.H, b = bh / c.H;
    mbar_arrive_expect_tx(c.bars + BAR_BDIN, TM * 128 + 2 * NHALF * 128);
    tma_load_4d(c.smem + OFF_QV, m_qv, c.bars + BAR_BDIN, h * DK, tile * TOUT, b, 0);
    tma_load_4d(c.smem + OFF_K, m_p, c.bars + BAR_BDIN, h * DK, 0, 0, 0);  // P -> K's buffer
    tma_load_4d(c.smem + OFF_K + NHALF * 128, m_p, c.bars + BAR_BDIN, h * DK, NHALF, 0, 0);
}
__device__ __forceinline__ uint32_t idesc_scores() {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(NHALF >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
}
// 128 x 320 x 64 score MMA: A = a 128 x 64 query tile at a_off, B = the two 160-row halves in K's buffer -> TMEM[0,320)
__device__ __noinline__ void ctl_score_mma(const Ctl& c, int a_off, int done_bar) {
    tc_fence_after();
    const uint32_t sa = smem_u32(c.smem + a_off), sb = smem_u32(c.smem + OFF_K);
#pragma unroll
    for (int nh = 0; nh < 2; ++nh)
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
            tc_mma_bf16(c.tmem_base + nh * NHALF, umma_desc(sa + kk * 32, 16, 1024), umma_desc(sb + nh * (NHALF * 128) + kk * 32, 16, 1024),
                        idesc_scores(), kk > 0 ? 1u : 0u);
    tc_commit(c.bars + done_bar);
}
__device__ __noinline__ void ctl_ac_loads(const Ctl& c, const CUtensorMap* m_qu, const CUtensorMap* m_k, int tt) {
    const int tile = tt % c.tiles, bh = tt / c.tiles;
    const int h = bh % c.H, b = bh / c.H;
    mbar_arrive_expect_tx(c.bars + BAR_ACIN, TM * 128 + 2 * NHALF * 128);
    tma_load_4d(c.smem + OFF_QU, m_qu, c.bars + BAR_ACIN, h * DK, tile * TOUT, b, 0);
    tma_load_4d(c.smem + OFF_K, m_k, c.bars + BAR_ACIN, h * DK, 0, b, 0);
    tma_load_4d(c.smem + OFF_K + NHALF * 128, m_k, c.bars + BAR_ACIN, h * DK, NHALF, b, 0);
}
// V of tile tt and, if there is one, (q+v) and P of tile tn: issued at the start of pass A (the shift before it is bound by
// shared-memory stores and should not share the port with 96 KB of TMA writes; V is not needed before p.V)
__device__ __noinline__ void ctl_v_next_loads(const Ctl& c, const CUtensorMap* m_v, const CUtensorMap* m_qv, const CUtensorMap* m_p, int tt,
                                              int tn) {
    const int bh = tt / c.tiles;
    const int h = bh % c.H, b = bh / c.H;
    mbar_arrive_expect_tx(c.bars + BAR_V, 5 * 8192);
    for (int kb = 0; kb < 5; ++kb) tma_load_4d(c.smem + OFF_P + kb * 8192, m_v, c.bars + BAR_V, h * DK, 64 * kb, b, 0);
    if (tn >= 0) ctl_bd_loads(c, m_qv, m_p, tn);
}
// O = p . V (K = keys, 16 per instruction; key blocks beyond T hold zero probabilities and are skipped) -> TMEM[320,384), then
// the bulk tensor stores of the probability tile: rows [r0, r0 + 127) x stored columns, straight from the MMA operand slabs
__device__ __noinline__ void ctl_pv_mma_store(const Ctl& c, const CUtensorMap* m_probs, int tt) {
    tc_fence_after();
    const uint32_t id_o = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((uint32_t)(DK >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
    const uint32_t s_stg = smem_u32(c.smem + OFF_STG), s_v = smem_u32(c.smem + OFF_P);
    const int ksteps = (c.T + 15) >> 4;
    for (int ks = 0; ks < ksteps; ++ks) {
        const int kb = ks >> 2, kk = ks & 3;
        tc_mma_bf16(c.tmem_base + TKMAX, umma_desc(s_stg + kb * (TM * 128) + kk * 32, 16, 1024),
                    umma_desc(s_v + kb * 8192 + kk * 2048, 8192, 1024), id_o, ks > 0 ? 1u : 0u);
    }
    tc_commit(c.bars + BAR_O_DONE);
    const int tile = tt % c.tiles, bh = tt / c.tiles;
    const int kslabs = (c.ld + 63) >> 6;
    for (int kb = 0; kb < kslabs; ++kb) tma_store_4d(m_probs, c.smem + OFF_STG + kb * (TM * 128), 64 * kb, tile * TOUT, bh, 0);
    bulk_commit();
}

// mask mode 4 (RAGGED): klen = lens[b] and the flat re-view runs over klen instead of T -- bd row r written at r (klen+1) + 1 + c
// for c < klen only (columns >= klen are products of real P rows here), shifted row read at r klen + j -- so that every valid
// row equals the batch-1 call on the utterance cut to klen frames.  Query rows >= klen drop the rel-pos term (their reads
// would reach flat positions no bd row of the tile wrote) and keep finite values.
__device__ __forceinline__ int ragged_len(const Params& p, int tt) {
    const long l = p.lens[(tt / p.tiles) / p.H];
    return (int)(l < p.T ? (l < 0 ? 0 : l) : p.T);
}

template <bool RAGGED>
__global__ void __launch_bounds__(THREADS, 1)
rel_attn_fwd_kernel(const __grid_constant__ CUtensorMap m_qu, const __grid_constant__ CUtensorMap m_qv,
                    const __grid_constant__ CUtensorMap m_k, const __grid_constant__ CUtensorMap m_v,
                    const __grid_constant__ CUtensorMap m_p, const __grid_constant__ CUtensorMap m_probs, const Params p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + OFF_BAR + 8 * NBARS);
    float* red = reinterpret_cast<float*>(smem + OFF_RED);  // [max | sum][column part][row]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int T = p.T;
    const int total = p.tiles * p.H * p.B;
    // The two single-thread roles (TMA producer, MMA issuer) are strictly sequential here, so ONE thread of an ordinary
    // worker warp plays both between its own phases: 16 warps = 4 per scheduler leave 128 registers per thread, which is what
    // keeps a warp's 80 score columns in registers without spills.
    const bool ctl = (warp == 0 && lane == 0);

    if (ctl) {
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&m_qu) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&m_qv) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&m_k) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&m_v) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&m_p) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&m_probs) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < NBARS; ++i)
            mbar_init(bars + i, (i == BAR_BD_DRAINED || i == BAR_P_READY || i == BAR_S_DRAINED || i == BAR_O_DRAINED) ? EPI_W : 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    Ctl cx;
    cx.smem = smem; cx.bars = bars; cx.tmem_base = tmem_base; cx.H = p.H; cx.tiles = p.tiles; cx.T = T; cx.ld = p.ld;

    const int q = warp & 3, part = warp >> 2;
    const int r = q * 32 + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    const float c2 = p.c2;
    const int cb = part * PARTW;
    uint16_t* flat = reinterpret_cast<uint16_t*>(smem + OFF_STG) + FLAT_PAD;

    // Persistent CTA: tiles blockIdx.x, + gridDim.x, ...  While the workers are in the softmax of tile n the control thread
    // already loads (q+v) and P of tile n + 1 (P into K's buffer, which the ac MMAs of tile n have released) and issues its bd
    // MMAs as soon as every warp has copied the scores of tile n out of TMEM, so that a tile starts with its shift: no load
    // or MMA latency, no CTA launch, no TMEM allocation on the per-tile path.  Every barrier completes once per tile:
    // parity = iteration & 1.
    if (ctl && (int)blockIdx.x < total) {
        ctl_bd_loads(cx, &m_qv, &m_p, blockIdx.x);
        mbar_wait(bars + BAR_BDIN, 0);
        ctl_score_mma(cx, OFF_QV, BAR_BD_DONE);  // bd = (q+v) . P^T
        // (q+u) and K (into P's place) once the bd MMAs have released it (later tiles: at the end of the previous tile)
        mbar_wait(bars + BAR_BD_DONE, 0);
        ctl_ac_loads(cx, &m_qu, &m_k, blockIdx.x);
    }
    __syncwarp();

    uint32_t ph = 0;
    for (int tt = blockIdx.x; tt < total; tt += gridDim.x, ph ^= 1u) {
        // (per-tile coordinates are recomputed where they are needed instead of living across the register-heavy passes)
        float sv[PARTW];  // the warp's 80 columns of its rows: bd, then scores, then exponentials
        FA_STAMP(0);

        // ---- shift: bd row g -> flat buffer (see the header comment)
        mbar_wait(bars + BAR_BD_DONE, ph);
        tc_fence_after();
        FA_STAMP(1);
        {
#pragma unroll
            for (int ch = 0; ch < PARTW / CH; ++ch) tc_ld16_issue(lane_addr + (uint32_t)(cb + ch * CH), sv + ch * CH);
            tc_wait_ld();
            FA_STAMP(12);
            // the flat buffer aliases the slabs the previous tile's probability stores read: they must be done (thread 0 issued
            // them) before anybody writes it; the barrier sits AFTER the TMEM reads so that it costs nothing
            if (ctl) bulk_wait_read<0>();
            __syncwarp();
            epi_barrier();
            FA_STAMP(2);
            const int r0 = (tt % p.tiles) * TOUT;
            const int W = RAGGED ? ragged_len(p, tt) : T;  // length the shift runs over
            const int off = r * (W + 1) + r0 - W;  // flat position of the padded zero of bd row g
            if (part == 0) flat[off] = 0;
            uint16_t* dst = flat + off + 1 + cb;
            // W odd: the row stride W + 1 is even, so every lane of the warp has the same 4-byte alignment and pairs of
            // halves go out as 32-bit stores (the phase is bound by shared-memory store wavefronts)
            const int par = (W & 1) ? ((off + 1 + cb) & 1) : 2;  // 0 aligned | 1 off by one half | 2 per-lane (scalar stores)
#pragma unroll
            for (int ch = 0; ch < PARTW / CH; ++ch) {
                const int c0 = cb + ch * CH;
                const float* v = sv + ch * CH;
                uint16_t* d = dst + ch * CH;
                if (c0 + CH <= W) {  // warp-uniform
                    if (par == 0) {
#pragma unroll
                        for (int e = 0; e < CH; e += 2) *reinterpret_cast<uint32_t*>(d + e) = f16x2_sat(v[e] * c2, v[e + 1] * c2);
                    } else if (par == 1) {
                        d[0] = (uint16_t)(f16x2_sat(v[0] * c2, 0.f) & 0xffffu);
#pragma unroll
                        for (int e = 1; e + 1 < CH; e += 2) *reinterpret_cast<uint32_t*>(d + e) = f16x2_sat(v[e] * c2, v[e + 1] * c2);
                        d[CH - 1] = (uint16_t)(f16x2_sat(v[CH - 1] * c2, 0.f) & 0xffffu);
                    } else {
#pragma unroll
                        for (int e = 0; e < CH; e += 2) {
                            const uint32_t h2 = f16x2_sat(v[e] * c2, v[e + 1] * c2);
                            d[e] = (uint16_t)(h2 & 0xffffu);
                            d[e + 1] = (uint16_t)(h2 >> 16);
                        }
                    }
                } else if (c0 < W) {  // columns >= W (zero products of the zero-filled P rows when W = T) must not reach the next row's slots
#pragma unroll
                    for (int e = 0; e < CH; e += 2) {
                        const uint32_t h2 = f16x2_sat(v[e] * c2, v[e + 1] * c2);
                        if (c0 + e < W) d[e] = (uint16_t)(h2 & 0xffffu);
                        if (c0 + e + 1 < W) d[e + 1] = (uint16_t)(h2 >> 16);
                    }
                }
            }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bars + BAR_BD_DRAINED);
        FA_STAMP(3);
        if (ctl) {  // ac = (q+u) . K^T into the same columns once every warp has copied its bd rows out
            mbar_wait(bars + BAR_ACIN, ph);
            mbar_wait(bars + BAR_BD_DRAINED, ph);
            ctl_score_mma(cx, OFF_QU, BAR_AC_DONE);
        }
        __syncwarp();
        epi_barrier();  // the flat buffer is complete
        FA_STAMP(4);

        // ---- pass A: s = ac * c2 + shifted bd, mask -- the warp's 80 columns stay in registers from here on; pass B:
        //      e = 2^(s - m) against the warp's OWN row maximum m, so that one exchange of (m, sum) per row part replaces a max
        //      round and a sum round: p = e * 2^(m - max_parts m) / sum_parts(sum * 2^(m - max))
        mbar_wait(bars + BAR_AC_DONE, ph);
        tc_fence_after();
        FA_STAMP(5);
        // the ac MMAs have released (q+u) and K's buffer: next tile's (q+v) and P; V of this tile (its buffer was released by the
        // previous tile's p.V, whose completion this thread has waited for as a worker).  A call: placed where no score column is live
        if (ctl) ctl_v_next_loads(cx, &m_v, &m_qv, &m_p, tt, tt + (int)gridDim.x < total ? tt + (int)gridDim.x : -1);
        __syncwarp();
        float mx = -INFINITY;
        {
#pragma unroll
            // (all 320 allocated columns are read unconditionally -- columns >= T are replaced below -- so that every element
            //  of sv is defined on every path and the array stays in registers)
            for (int ch = 0; ch < PARTW / CH; ++ch) tc_ld16_issue(lane_addr + (uint32_t)(cb + ch * CH), sv + ch * CH);
            tc_wait_ld();
            FA_STAMP(13);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bars + BAR_S_DRAINED);  // TMEM[0,320) may take the next tile's bd
            // shifted row r starts at half r T + cb of the flat buffer: aligned 32-bit loads from the word below and a funnel
            // shift by the lane's own parity (row stride T may be odd) instead of 16-bit loads
            int klen = T;
            if (RAGGED) {
                klen = ragged_len(p, tt);
            } else if (p.mask_mode != 0 && p.lens) {
                const long l = p.lens[(tt / p.tiles) / p.H];
                long k = l;
                if (p.mask_mode == 2) k = l + 1;
                else if (p.mask_mode == 3) k = (l + 3) / 4;
                klen = (int)(k < T ? (k < 0 ? 0 : k) : T);
            }
            const int h0 = r * (RAGGED ? klen : T) + cb;
            const bool qpad = RAGGED && (tt % p.tiles) * TOUT + r >= klen;  // padded query row: no rel-pos term
            const int fpar = h0 & 1;
            const uint32_t* src = reinterpret_cast<const uint32_t*>(flat + (h0 - fpar));
            const uint32_t fsh = 16u * (uint32_t)fpar;
#pragma unroll
            for (int ch = 0; ch < PARTW / CH; ++ch) {
                const int j0 = cb + ch * CH;
                float* v = sv + ch * CH;
                uint32_t w[CH / 2 + 1];
#pragma unroll
                for (int k = 0; k <= CH / 2; ++k) w[k] = src[ch * (CH / 2) + k];
                const bool clean = j0 + CH <= klen;  // no masked or padding column in this chunk (warp-uniform)
#pragma unroll
                for (int k = 0; k < CH / 2; ++k) {
                    const uint32_t pr = __funnelshift_r(w[k], w[k + 1], fsh);
                    float2 f = __half22float2(*reinterpret_cast<const __half2*>(&pr));
                    if (RAGGED && qpad) f = make_float2(0.f, 0.f);
                    float s0 = fmaf(v[2 * k], c2, f.x), s1 = fmaf(v[2 * k + 1], c2, f.y);
                    if (!clean) {
                        const int j = j0 + 2 * k;
                        s0 = (j < klen) ? s0 : -1e38f;
                        s0 = (j < T) ? s0 : -INFINITY;
                        s1 = (j + 1 < klen) ? s1 : -1e38f;
                        s1 = (j + 1 < T) ? s1 : -INFINITY;
                    }
                    v[2 * k] = s0;
                    v[2 * k + 1] = s1;
                    mx = fmaxf(mx, fmaxf(s0, s1));
                }
            }
        }
        FA_STAMP(6);
        const float mloc = (mx == -INFINITY) ? 0.f : mx;  // a part that lies entirely beyond T contributes nothing
        float sum = 0.f;
#pragma unroll
        for (int e = 0; e < PARTW; ++e) {
            sv[e] = ex2_fast(sv[e] - mloc);
            sum += sv[e];
        }
        red[part * TM + r] = mx;
        red[4 * TM + part * TM + r] = sum;
        FA_STAMP(7);
        epi_barrier();
        FA_STAMP(8);
        float inv;
        {
            const float m0 = red[r], m1 = red[TM + r], m2 = red[2 * TM + r], m3 = red[3 * TM + r];
            const float mall = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));  // finite: column 0 exists and masked scores are -1e38
            const float tot = red[4 * TM + r] * ex2_fast(m0 - mall) + red[5 * TM + r] * ex2_fast(m1 - mall) +
                              red[6 * TM + r] * ex2_fast(m2 - mall) + red[7 * TM + r] * ex2_fast(m3 - mall);
            inv = __fdividef(ex2_fast(mloc - mall), tot);
        }

        // ---- pass C: p = e * inv -> bf16 -> K-major SWIZZLE_128B slabs (element (r, j): slab j / 64, row r, 16-byte chunk
        //      ((j % 64) / 8) ^ (r % 8)): the layout TMA produces for a {64, 128} box, which the MMA and the stores consume
#pragma unroll
        for (int ch = 0; ch < PARTW / CH; ++ch) {
            const int j0 = cb + ch * CH;
            if (j0 < p.ld) {  // every stored column: [T, ld) holds exact zeros (e = 2^-inf)
                const float* v = sv + ch * CH;
                uint8_t* rowp = smem + OFF_STG + (j0 >> 6) * (TM * 128) + r * 128;
                const int ch0 = (j0 & 63) >> 3;
#pragma unroll
                for (int t = 0; t < CH / 8; ++t) {
                    uint4 u;
                    u.x = pack2(v[8 * t] * inv, v[8 * t + 1] * inv);
                    u.y = pack2(v[8 * t + 2] * inv, v[8 * t + 3] * inv);
                    u.z = pack2(v[8 * t + 4] * inv, v[8 * t + 5] * inv);
                    u.w = pack2(v[8 * t + 6] * inv, v[8 * t + 7] * inv);
                    *reinterpret_cast<uint4*>(rowp + (((ch0 + t) ^ (r & 7)) << 4)) = u;
                }
            }
        }
        fence_proxy_async();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bars + BAR_P_READY);
        FA_STAMP(9);
        if (ctl) {
            // O = p . V  (K = keys, 16 per instruction; key blocks beyond T hold zero probabilities and are skipped)
            const bool has_next = tt + (int)gridDim.x < total;
            if (has_next) {  // the next tile's bd first: every warp has copied this tile's scores out of TMEM[0,320)
                mbar_wait(bars + BAR_S_DRAINED, ph);
                mbar_wait(bars + BAR_BDIN, ph ^ 1);
                ctl_score_mma(cx, OFF_QV, BAR_BD_DONE);
            }
            mbar_wait(bars + BAR_V, ph);
            mbar_wait(bars + BAR_P_READY, ph);
            if (tt != (int)blockIdx.x) mbar_wait(bars + BAR_O_DRAINED, ph ^ 1);  // the workers have read the previous tile's O out of TMEM
            ctl_pv_mma_store(cx, &m_probs, tt);
            if (has_next) {
                // the next tile's (q+u) and K as soon as its bd MMAs have released P: the 56 KB land while this tile's O is
                // stored, not during the next shift (which is bound by shared-memory store wavefronts)
                mbar_wait(bars + BAR_BD_DONE, ph ^ 1);
                ctl_ac_loads(cx, &m_qu, &m_k, tt + gridDim.x);
            }
        }
        __syncwarp();

        // ---- O tile: this warp's 32 rows x 16 of the 64 head columns
        mbar_wait(bars + BAR_O_DONE, ph);
        tc_fence_after();
        FA_STAMP(10);
        {
            float v[CH];
            tc_ld16(lane_addr + (uint32_t)(TKMAX + CH * part), v);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bars + BAR_O_DRAINED);
            const int tile = tt % p.tiles, bh = tt / p.tiles;
            const int h = bh % p.H, b = bh / p.H, g = tile * TOUT + r;
            if (r < TOUT && g < T) {
                uint4* dst = reinterpret_cast<uint4*>(p.o + ((long)b * T + g) * p.ldo + h * DK + CH * part);
#pragma unroll
                for (int t = 0; t < CH / 8; ++t) {
                    uint4 u;
                    u.x = pack2(v[8 * t], v[8 * t + 1]);
                    u.y = pack2(v[8 * t + 2], v[8 * t + 3]);
                    u.z = pack2(v[8 * t + 4], v[8 * t + 5]);
                    u.w = pack2(v[8 * t + 6], v[8 * t + 7]);
                    dst[t] = u;
                }
            }
        }
        FA_STAMP(11);
    }
    if (ctl) bulk_wait_read<0>();  // the probability tile must outlive the bulk stores that read it
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
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

// bf16 tensor (batch, rows, inner) with element strides (sbatch, ld, 1); box {64 inner, box_rows}
static int make_map(CUtensorMap* map, const void* base, long inner, long rows, long ld, long nbatch, long sbatch, int box_rows,
                    bool store) {
    auto enc = encoder();
    if (!enc) { set_error("cuTensorMapEncodeTiled entry point unavailable"); return LASR_ERR_DRIVER; }
    const cuuint64_t row_bytes = (cuuint64_t)ld * 2;
    const bool useb = nbatch > 1 && sbatch != 0;
    cuuint64_t dims[4] = {(cuuint64_t)inner, (cuuint64_t)rows, (cuuint64_t)(useb ? nbatch : 1), 1};
    cuuint64_t strides[3] = {row_bytes, useb ? (cuuint64_t)sbatch * 2 : row_bytes, useb ? (cuuint64_t)sbatch * 2 : row_bytes};
    cuuint32_t box[4] = {64, (cuuint32_t)box_rows, 1, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (strides[0] & 15) || (strides[1] & 15)) {
        set_error("rel_attn_fwd: operand base/strides must be 16-byte aligned (base=%p ld=%ld batch stride=%ld)", base, ld, sbatch);
        return LASR_ERR_BAD_ARG;
    }
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                     store ? CU_TENSOR_MAP_L2_PROMOTION_NONE : CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("rel_attn_fwd: cuTensorMapEncodeTiled failed (%d): inner=%ld rows=%ld ld=%ld", (int)r, inner, rows, ld);
        return LASR_ERR_DRIVER;
    }
    return LASR_OK;
}

}  // namespace fa
}  // namespace lasr

extern "C" {
using namespace lasr;

static long long* g_fa_trace = nullptr;
/* developer aid: device buffer of 16 int64 per CTA that receives clock64 stamps of the kernel's phases (NULL = off) */
void lasr_rel_attn_fwd_set_trace(void* buf) { g_fa_trace = reinterpret_cast<long long*>(buf); }

int lasr_rel_attn_fwd_supported(int T, int dk) { return (T >= 1 && T <= fa::TKMAX && dk == fa::DK) ? 1 : 0; }

int lasr_rel_attn_fwd(const void* qu, const void* qv, long ldq, const void* k, const void* v, long ldkv, const void* pos, long ldp,
                      void* probs, int ld, void* o, long ldo, const int64_t* lens, int mask_mode, float scale, int B, int H, int T,
                      int dk, void* stream) {
    LASR_REQUIRE(qu && qv && k && v && pos && probs && o && B > 0 && H > 0, "rel_attn_fwd: null operand or empty batch");
    if (!lasr_rel_attn_fwd_supported(T, dk)) {
        set_error("rel_attn_fwd: needs 1 <= T <= %d and dk == %d (got T=%d dk=%d)", fa::TKMAX, fa::DK, T, dk);
        return LASR_ERR_UNSUPPORTED;
    }
    LASR_REQUIRE(ld >= T && ld % 8 == 0 && ld <= fa::TKMAX, "rel_attn_fwd: ld must be a multiple of 8 in [T, %d]", fa::TKMAX);
    LASR_REQUIRE(mask_mode >= 0 && mask_mode <= 4 && (mask_mode == 0 || lens), "rel_attn_fwd: bad mask mode");
    LASR_REQUIRE(ldo % 8 == 0 && (reinterpret_cast<uintptr_t>(o) & 15) == 0 && (reinterpret_cast<uintptr_t>(probs) & 15) == 0,
                 "rel_attn_fwd: O and probs must be 16-byte aligned");
    const long d = (long)H * dk;
    CUtensorMap m_qu, m_qv, m_k, m_v, m_p, m_probs;
    int rc;
    if ((rc = fa::make_map(&m_qu, qu, d, T, ldq, B, (long)T * ldq, fa::TM, false)) != LASR_OK) return rc;
    if ((rc = fa::make_map(&m_qv, qv, d, T, ldq, B, (long)T * ldq, fa::TM, false)) != LASR_OK) return rc;
    if ((rc = fa::make_map(&m_k, k, d, T, ldkv, B, (long)T * ldkv, fa::NHALF, false)) != LASR_OK) return rc;
    if ((rc = fa::make_map(&m_v, v, d, T, ldkv, B, (long)T * ldkv, 64, false)) != LASR_OK) return rc;
    if ((rc = fa::make_map(&m_p, pos, d, T, ldp, 1, 0, fa::NHALF, false)) != LASR_OK) return rc;
    if ((rc = fa::make_map(&m_probs, probs, ld, T, ld, (long)B * H, (long)T * ld, fa::TOUT, true)) != LASR_OK) return rc;
    static bool configured = false;
    if (!configured) {
        if (cudaFuncSetAttribute(fa::rel_attn_fwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, fa::SMEM_BYTES) != cudaSuccess ||
            cudaFuncSetAttribute(fa::rel_attn_fwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, fa::SMEM_BYTES) != cudaSuccess)
            return check_launch("rel_attn_fwd smem attr");
        configured = true;
    }
    fa::Params p;
    p.o = reinterpret_cast<bf16*>(o);
    p.ldo = ldo;
    p.lens = lens;
    p.mask_mode = mask_mode;
    p.c2 = scale * 1.4426950408889634f;
    p.B = B; p.H = H; p.T = T; p.ld = ld;
    p.tiles = (T + fa::TOUT - 1) / fa::TOUT;
    p.trace = g_fa_trace;
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
    }
    const long total = (long)p.tiles * H * B;
    const int grid = (int)(total < sms ? total : sms);  // persistent: one CTA per SM walks the (batch, head, row tile) list
    if (mask_mode == 4)
        launch_pdl(fa::rel_attn_fwd_kernel<true>, dim3((unsigned)grid), dim3(fa::THREADS), (size_t)fa::SMEM_BYTES,
                   (cudaStream_t)stream, m_qu, m_qv, m_k, m_v, m_p, m_probs, p);
    else
        launch_pdl(fa::rel_attn_fwd_kernel<false>, dim3((unsigned)grid), dim3(fa::THREADS), (size_t)fa::SMEM_BYTES,
                   (cudaStream_t)stream, m_qu, m_qv, m_k, m_v, m_p, m_probs, p);
    return check_launch("rel_attn_fwd");
}

}  // extern "C"
