// Inference-side pieces of the path (models/u2.py:221-317, nets/ctc.py:25-26):
//   lasr_logsoftmax_topk        (device) per frame: log-sum-exp, optional full log-softmax, and the K best classes in
//                               (log-prob descending, index ascending) order -- the `torch.topk(logp, beam)` prune of the
//                               CTC prefix beam search (u2.py:230) and, with K = 1, greedy CTC's argmax.
//   lasr_gather_logp            (device) logp[row, tok[row]] = logits[row, tok] - lse[row]: the attention-rescoring lookups
//                               (u2.py:306-310) without materialising the (beam, L, V) log-softmax.
//   lasr_ctc_prefix_beam_search (HOST)   the prefix search itself (u2.py:224-261) on the pruned (frames, K) matrix.  It is a
//                               sequential dictionary algorithm in float64 Python arithmetic in the reference; it is restated
//                               here in C++ with the same operation order (libm exp/log, left-to-right sums, insertion-ordered
//                               map, stable sort), so n-best lists and scores are bit-identical given the same log-probs.
//   lasr_ctc_prefix_beam_search_batch (device) the same search for a ragged batch in one launch, one warp per utterance;
//                               float64 with CUDA's exp / log, so scores may differ from the host's in the last bits.
#include <cmath>
#include <cstring>
#include <algorithm>
#include <limits>
#include <string>
#include <unordered_map>
#include <vector>

#include <math_constants.h>

#include "common.cuh"

namespace lasr {

// ---------------------------------------------------------------------------------------------
// log-softmax + top-K: one CTA (256 threads) per row
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) logsoftmax_topk_kernel(const T* __restrict__ logits, long ld, int V, int K,
                                                              float* __restrict__ lse_out, float* __restrict__ logp_full, long ldf,
                                                              float* __restrict__ top_val, int* __restrict__ top_idx) {
    __shared__ float scratch[32];
    __shared__ float sv[8];
    __shared__ int si[8];
    const long row = blockIdx.x;
    const T* x = logits + row * ld;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float mx = -INFINITY;
    for (int c = threadIdx.x; c < V; c += 256) mx = fmaxf(mx, to_f32<T>(x[c]));
    mx = block_max(mx, scratch);
    float sum = 0.f;
    for (int c = threadIdx.x; c < V; c += 256) sum += expf(to_f32<T>(x[c]) - mx);
    sum = block_sum(sum, scratch);
    const float lsum = logf(sum);
    if (threadIdx.x == 0 && lse_out) lse_out[row] = mx + lsum;
    // log-probabilities are formed as (x - max) - log(sum), the rounding sequence of torch.log_softmax: the reference ranks the
    // ROUNDED fp32 log-probs (argmax / torch.topk of log_softmax), where two classes whose logits differ in the last bits can tie
    if (logp_full)
        for (int c = threadIdx.x; c < V; c += 256) logp_full[row * ldf + c] = (to_f32<T>(x[c]) - mx) - lsum;
    // K rounds of arg-max in the total order (log-prob descending, index ascending); round r only considers elements that come
    // strictly after the previous winner in that order, so no "taken" set is needed
    float last_v = INFINITY;
    int last_i = -1;
    for (int r = 0; r < K; ++r) {
        float bv = -INFINITY;
        int bi = 0x7fffffff;
        for (int c = threadIdx.x; c < V; c += 256) {
            const float v = (to_f32<T>(x[c]) - mx) - lsum;
            const bool after = (v < last_v) || (v == last_v && c > last_i);
            if (after && (v > bv || (v == bv && c < bi))) { bv = v; bi = c; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
        }
        __syncthreads();
        if (lane == 0) { sv[warp] = bv; si[warp] = bi; }
        __syncthreads();
        bv = sv[0]; bi = si[0];
#pragma unroll
        for (int w = 1; w < 8; ++w)
            if (sv[w] > bv || (sv[w] == bv && si[w] < bi)) { bv = sv[w]; bi = si[w]; }
        if (threadIdx.x == 0) {
            top_val[row * K + r] = (bi == 0x7fffffff) ? -INFINITY : bv;
            top_idx[row * K + r] = (bi == 0x7fffffff) ? -1 : bi;
        }
        last_v = bv;
        last_i = bi;
    }
}

template <typename T>
__global__ void __launch_bounds__(256) gather_logp_kernel(const T* __restrict__ logits, long ld, const float* __restrict__ lse,
                                                          const int64_t* __restrict__ tok, float* __restrict__ out, long rows, int V) {
    const long r = (long)blockIdx.x * 256 + threadIdx.x;
    if (r >= rows) return;
    const long t = tok[r];
    out[r] = (t >= 0 && t < V) ? to_f32<T>(logits[r * ld + t]) - lse[r] : 0.f;
}

// ---------------------------------------------------------------------------------------------
// host: CTC prefix beam search
// ---------------------------------------------------------------------------------------------
static const double NINF = -std::numeric_limits<double>::infinity();

// models/u2.py:367-375
static double log_add(const double* a, int n) {
    bool all_inf = true;
    for (int i = 0; i < n; ++i) all_inf = all_inf && (a[i] == NINF);
    if (all_inf) return NINF;
    double a_max = a[0];
    for (int i = 1; i < n; ++i) a_max = std::max(a_max, a[i]);
    double s = 0.0;
    for (int i = 0; i < n; ++i) s += std::exp(a[i] - a_max);
    return a_max + std::log(s);
}

struct Hyp {
    std::vector<int32_t> prefix;
    double pb, pnb;
};

static std::string key_of(const std::vector<int32_t>& p) {
    return std::string(reinterpret_cast<const char*>(p.data()), p.size() * sizeof(int32_t));
}

// ---------------------------------------------------------------------------------------------
// device: CTC prefix beam search over a ragged batch, one warp (one CTA) per utterance
// ---------------------------------------------------------------------------------------------
// The host function below restated operation for operation.  A prefix is a node (parent, token) of a per-utterance pool; only
// hypotheses that survive a prune get one, at id t * beam + rank.  Per frame:
//   1. contributions in the host's loop order (j over the K classes, h over the beam), placed by a warp scan: each carries the
//      key of the entry it updates -- h' < beam for a prefix already in the beam (h itself, or h' = h + s when such a
//      hypothesis exists), beam + pair for a new extension (top_idx holds distinct classes, so those are all distinct)
//   2. lane h' folds the contributions of key h' in loop order through the same log_add; an extension has one contribution
//   3. entries are numbered by first touch; rank = stable descending sort by log_add(pb, pnb); rank < beam survives
// Exact arithmetic: float64 with CUDA's exp / log (<= 1 ulp, not glibc's), so scores may differ from the host's in the last
// bits and two hypotheses within a few ulps of each other may swap.
constexpr int PB_MAX_BEAM = 32, PB_MAX_K = 64;

// log_add of (a0, a1) or (a0, a1, a2): the host's operation order with scalar arguments (no local-memory array)
__device__ __forceinline__ double log_add_d(double a0, double a1, double a2, bool three) {
    const double ninf = -CUDART_INF;
    if (a0 == ninf && a1 == ninf && (!three || a2 == ninf)) return ninf;
    double a_max = fmax(a0, a1);
    if (three) a_max = fmax(a_max, a2);
    double s = 0.0;
    s += exp(a0 - a_max);
    s += exp(a1 - a_max);
    if (three) s += exp(a2 - a_max);
    return a_max + log(s);
}

struct PbBeam {  // one hypothesis of the beam
    double pb, pnb;
    int node, len, last;  // node -1 = empty prefix; last = its final token (-1 if empty)
};

// Shared-memory layout of one CTA (sizes from K and beam)
struct PbSmem {
    PbBeam* cur;
    PbBeam* nxt;
    int* ckey;       // [2 K beam]  entry key of a contribution
    int* cmeta;      // [2 K beam]  field (bit 0: 0 pb / 1 pnb) | term count (bit 1: 3 terms) | pair index << 2
    double* cterm;   // [2 K beam][2]
    int* cflag;      // [2 K beam]  entry id of a first touch, -1 otherwise
    double* ev;      // [K beam + beam][3]  pb, pnb, score of each entry
    int* ekey;       // [K beam + beam]     key of the entry, and the contribution that created it (new extensions)
    int* esrc;
};

__host__ __device__ inline size_t pb_smem_bytes(int K, int beam) {
    const size_t nc = 2 * (size_t)K * beam, ne = (size_t)K * beam + beam;
    return 2 * beam * sizeof(PbBeam) + nc * (3 * sizeof(int) + 2 * sizeof(double)) + ne * (3 * sizeof(double) + 2 * sizeof(int)) + 64;
}

// prefix(a) == prefix(b) for two nodes of equal length: equal ids end the walk (a prefix can own two nodes when it was pruned
// and re-created while one of its extensions survived)
__device__ __forceinline__ bool same_prefix(const int2* pool, int a, int b) {
    while (a != b) {
        if (a < 0 || b < 0) return false;
        const int2 na = pool[a], nb = pool[b];
        if (na.y != nb.y) return false;
        a = na.x;
        b = nb.x;
    }
    return true;
}

__global__ void __launch_bounds__(32) ctc_prefix_beam_search_kernel(const float* __restrict__ top_val, const int* __restrict__ top_idx,
                                                                    const int64_t* __restrict__ frames, int Tmax, int K, int beam,
                                                                    int blank, int2* __restrict__ pool_all, int32_t* __restrict__ out_tokens,
                                                                    int32_t* __restrict__ out_lens, double* __restrict__ out_scores,
                                                                    int32_t* __restrict__ out_n, int max_len) {
    extern __shared__ __align__(16) uint8_t pb_raw[];
    const int b = blockIdx.x, lane = threadIdx.x;
    const int nc_max = 2 * K * beam, ne_max = K * beam + beam;
    PbSmem S;
    {
        uint8_t* p = pb_raw;
        S.cur = reinterpret_cast<PbBeam*>(p); p += beam * sizeof(PbBeam);
        S.nxt = reinterpret_cast<PbBeam*>(p); p += beam * sizeof(PbBeam);
        S.cterm = reinterpret_cast<double*>(p); p += (size_t)nc_max * 2 * sizeof(double);
        S.ev = reinterpret_cast<double*>(p); p += (size_t)ne_max * 3 * sizeof(double);
        S.ckey = reinterpret_cast<int*>(p); p += nc_max * sizeof(int);
        S.cmeta = reinterpret_cast<int*>(p); p += nc_max * sizeof(int);
        S.cflag = reinterpret_cast<int*>(p); p += nc_max * sizeof(int);
        S.ekey = reinterpret_cast<int*>(p); p += ne_max * sizeof(int);
        S.esrc = reinterpret_cast<int*>(p);
    }
    long nf = frames[b];
    nf = nf < 0 ? 0 : (nf > Tmax ? Tmax : nf);
    int2* pool = pool_all + (long)b * Tmax * beam;
    const float* tv = top_val + (long)b * Tmax * K;
    const int* ti = top_idx + (long)b * Tmax * K;
    if (lane == 0) S.cur[0] = PbBeam{0.0, -CUDART_INF, -1, 0, -1};
    int nh = 1;
    __syncwarp();
    for (int t = 0; t < nf; ++t) {
        // ---- 1. contributions in loop order
        const int npairs = K * nh;
        int nc = 0;
        for (int q0 = 0; q0 < npairs; q0 += 32) {
            const int q = q0 + lane;
            int cnt = 0, s = -1, h = 0;
            double ps = 0.0;
            if (q < npairs) {
                const int j = q / nh;
                h = q - j * nh;
                s = ti[(long)t * K + j];
                ps = (double)tv[(long)t * K + j];
                if (s >= 0) cnt = (s != blank && s == S.cur[h].last) ? 2 : 1;
            }
            int incl = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += v;
            }
            int pos = nc + incl - cnt;
            if (cnt > 0) {
                const PbBeam hy = S.cur[h];
                if (s == blank) {  // *  -> *   (pb)
                    S.ckey[pos] = h; S.cmeta[pos] = 0 | 2 | (q << 2);
                    S.cterm[2 * pos] = hy.pb + ps; S.cterm[2 * pos + 1] = hy.pnb + ps;
                } else {
                    if (cnt == 2) {  // *s -> *s  (pnb)
                        S.ckey[pos] = h; S.cmeta[pos] = 1 | (q << 2);
                        S.cterm[2 * pos] = hy.pnb + ps;
                        ++pos;
                    }
                    // the extension prefix(h) + s: a hypothesis of the beam already, or a new entry
                    int key = beam + q;
                    for (int h2 = 0; h2 < nh; ++h2) {
                        const PbBeam& o = S.cur[h2];
                        if (o.len == hy.len + 1 && o.last == s && same_prefix(pool, pool[o.node].x, hy.node)) { key = h2; break; }
                    }
                    S.ckey[pos] = key;
                    if (cnt == 2) {  // *s-s -> *ss  (pnb, two terms)
                        S.cmeta[pos] = 1 | (q << 2);
                        S.cterm[2 * pos] = hy.pb + ps;
                    } else {         // *  -> *s  (pnb, three terms)
                        S.cmeta[pos] = 1 | 2 | (q << 2);
                        S.cterm[2 * pos] = hy.pb + ps; S.cterm[2 * pos + 1] = hy.pnb + ps;
                    }
                }
            }
            nc += __shfl_sync(0xffffffffu, incl, 31);
        }
        __syncwarp();
        // ---- 2. folds in loop order: lane h' for the beam's own prefixes, any lane for a new extension
        double fpb = -CUDART_INF, fpnb = -CUDART_INF;
        int first = 0x7fffffff;
        if (lane < nh) {
            for (int c = 0; c < nc; ++c) {
                if (S.ckey[c] != lane) continue;
                first = min(first, c);
                const int m = S.cmeta[c];
                const double r = log_add_d((m & 1) ? fpnb : fpb, S.cterm[2 * c], S.cterm[2 * c + 1], (m & 2) != 0);
                if (m & 1) fpnb = r; else fpb = r;
            }
        }
        for (int c = lane; c < nc; c += 32) S.cflag[c] = S.ckey[c] >= beam ? 1 : 0;
        __syncwarp();
        if (lane < nh && first != 0x7fffffff) S.cflag[first] = 1;
        __syncwarp();
        // entry ids = scan of the first-touch flags
        int ne = 0;
        for (int c0 = 0; c0 < nc; c0 += 32) {
            const int c = c0 + lane;
            const int f = c < nc ? S.cflag[c] : 0;
            int incl = f;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += v;
            }
            if (f) {
                const int e = ne + incl - 1;
                const int key = S.ckey[c];
                S.ekey[e] = key;
                S.esrc[e] = c;
                if (key >= beam) {
                    const int m = S.cmeta[c];
                    S.ev[3 * e] = -CUDART_INF;
                    S.ev[3 * e + 1] = log_add_d(-CUDART_INF, S.cterm[2 * c], S.cterm[2 * c + 1], (m & 2) != 0);
                }
            }
            ne += __shfl_sync(0xffffffffu, incl, 31);
        }
        __syncwarp();
        // the folds of the beam's own prefixes live in lanes h': publish them at the entry of their first touch
        if (lane < nh && first != 0x7fffffff) {
            int e = 0;
            for (; e < ne; ++e) if (S.esrc[e] == first) break;
            S.ev[3 * e] = fpb;
            S.ev[3 * e + 1] = fpnb;
        }
        __syncwarp();
        for (int e = lane; e < ne; e += 32) {
            S.ev[3 * e + 2] = log_add_d(S.ev[3 * e], S.ev[3 * e + 1], 0.0, false);
        }
        __syncwarp();
        // ---- 3. stable descending sort by score (ties: first touch first); the best `beam` survive
        const int nkeep = min(beam, ne);
        for (int e = lane; e < ne; e += 32) {
            const double sc = S.ev[3 * e + 2];
            int rank = 0;
            for (int e2 = 0; e2 < ne && rank < beam; ++e2) {
                const double s2 = S.ev[3 * e2 + 2];
                rank += (s2 > sc || (s2 == sc && e2 < e)) ? 1 : 0;
            }
            if (rank < beam) {
                const int key = S.ekey[e];
                PbBeam nh_;
                nh_.pb = S.ev[3 * e];
                nh_.pnb = S.ev[3 * e + 1];
                if (key < beam) {
                    const PbBeam& o = S.cur[key];
                    nh_.node = o.node; nh_.len = o.len; nh_.last = o.last;
                } else {
                    const int q = S.cmeta[S.esrc[e]] >> 2;
                    const int j = q / nh, h = q - j * nh;
                    const int s = ti[(long)t * K + j];
                    const int id = t * beam + rank;
                    pool[id] = make_int2(S.cur[h].node, s);
                    nh_.node = id; nh_.len = S.cur[h].len + 1; nh_.last = s;
                }
                S.nxt[rank] = nh_;
            }
        }
        __syncwarp();
        for (int i = lane; i < nkeep; i += 32) S.cur[i] = S.nxt[i];
        nh = nkeep;
        __syncwarp();
    }
    // ---- output: tokens by walking the parent links
    for (int i = lane; i < beam; i += 32) {
        int32_t* row = out_tokens + ((long)b * beam + i) * max_len;
        if (i < nh) {
            const PbBeam hy = S.cur[i];
            const int len = min(hy.len, max_len);
            for (int j = len; j < max_len; ++j) row[j] = -1;
            int nd = hy.node;
            for (int j = hy.len - 1; j >= 0; --j) {
                const int2 n = pool[nd];
                if (j < max_len) row[j] = n.y;
                nd = n.x;
            }
            out_lens[(long)b * beam + i] = hy.len;
            out_scores[(long)b * beam + i] = log_add_d(hy.pb, hy.pnb, 0.0, false);
        } else {
            for (int j = 0; j < max_len; ++j) row[j] = -1;
            out_lens[(long)b * beam + i] = 0;
            out_scores[(long)b * beam + i] = -CUDART_INF;
        }
    }
    if (lane == 0) out_n[b] = nh;
}

}  // namespace lasr

extern "C" {
using namespace lasr;

int lasr_logsoftmax_topk(const void* logits, int dtype, int64_t ld, int64_t rows, int V, int K, float* lse, float* logp_full,
                         int64_t ldf, float* top_val, int32_t* top_idx, void* stream) {
    LASR_REQUIRE(logits && rows > 0 && V > 0 && K >= 0 && (K == 0 || (top_val && top_idx)) && K <= V, "logsoftmax_topk: bad args");
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == LASR_F32) logsoftmax_topk_kernel<float><<<(unsigned)rows, 256, 0, st>>>((const float*)logits, ld, V, K, lse, logp_full, ldf, top_val, top_idx);
    else if (dtype == LASR_BF16) logsoftmax_topk_kernel<bf16><<<(unsigned)rows, 256, 0, st>>>((const bf16*)logits, ld, V, K, lse, logp_full, ldf, top_val, top_idx);
    else { set_error("logsoftmax_topk: bad dtype"); return LASR_ERR_UNSUPPORTED; }
    return check_launch("logsoftmax_topk");
}

int lasr_gather_logp(const void* logits, int dtype, int64_t ld, const float* lse, const int64_t* tokens, float* out, int64_t rows, int V,
                     void* stream) {
    LASR_REQUIRE(logits && lse && tokens && out && rows > 0 && V > 0, "gather_logp: bad args");
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == LASR_F32) gather_logp_kernel<float><<<ceil_div(rows, 256), 256, 0, st>>>((const float*)logits, ld, lse, tokens, out, rows, V);
    else if (dtype == LASR_BF16) gather_logp_kernel<bf16><<<ceil_div(rows, 256), 256, 0, st>>>((const bf16*)logits, ld, lse, tokens, out, rows, V);
    else { set_error("gather_logp: bad dtype"); return LASR_ERR_UNSUPPORTED; }
    return check_launch("gather_logp");
}

size_t lasr_ctc_prefix_beam_search_batch_workspace(int B, int Tmax, int beam) {
    return (B > 0 && Tmax > 0 && beam > 0) ? (size_t)B * Tmax * beam * sizeof(int2) : 0;
}

int lasr_ctc_prefix_beam_search_batch(const float* top_val, const int32_t* top_idx, const int64_t* frames, int B, int Tmax, int K, int beam,
                                      int blank, int32_t* out_tokens, int32_t* out_lens, double* out_scores, int32_t* out_n, int max_len,
                                      void* workspace, size_t ws_bytes, void* stream) {
    LASR_REQUIRE(top_val && top_idx && frames && out_tokens && out_lens && out_scores && out_n && B > 0 && Tmax > 0 && max_len >= Tmax,
                 "ctc_prefix_beam_search_batch: bad args (max_len must be >= Tmax)");
    LASR_REQUIRE(K >= 1 && K <= PB_MAX_K && beam >= 1 && beam <= PB_MAX_BEAM, "ctc_prefix_beam_search_batch: needs 1 <= K <= %d, 1 <= beam <= %d",
                 PB_MAX_K, PB_MAX_BEAM);
    LASR_REQUIRE(workspace && ws_bytes >= lasr_ctc_prefix_beam_search_batch_workspace(B, Tmax, beam),
                 "ctc_prefix_beam_search_batch: workspace too small");
    const size_t smem = pb_smem_bytes(K, beam);
    if (smem > 48 * 1024 &&
        cudaFuncSetAttribute(ctc_prefix_beam_search_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
        return check_launch("ctc_prefix_beam_search_batch smem attr");
    ctc_prefix_beam_search_kernel<<<B, 32, smem, (cudaStream_t)stream>>>(top_val, top_idx, frames, Tmax, K, beam, blank, (int2*)workspace,
                                                                         out_tokens, out_lens, out_scores, out_n, max_len);
    return check_launch("ctc_prefix_beam_search_batch");
}

/* HOST function: topk_logp / topk_idx are host arrays (frames, K), row-major, classes in the order the device kernel emits
 * (log-prob descending).  Writes up to `beam` hypotheses best first: tokens (beam, max_len) padded with -1, lengths, scores
 * (= log_add(p_blank, p_nonblank) in float64).  *n_out = number of hypotheses. */
int lasr_ctc_prefix_beam_search(const float* topk_logp, const int32_t* topk_idx, int frames, int K, int beam, int blank,
                                int32_t* out_tokens, int32_t* out_lens, double* out_scores, int max_len, int32_t* n_out) {
    LASR_REQUIRE(topk_logp && topk_idx && out_tokens && out_lens && out_scores && n_out && frames >= 0 && K > 0 && beam > 0 && max_len >= 0,
                 "ctc_prefix_beam_search: bad args");
    std::vector<Hyp> cur(1);
    cur[0].pb = 0.0;
    cur[0].pnb = NINF;
    std::vector<Hyp> next;
    std::unordered_map<std::string, int> index;
    std::vector<std::pair<double, int>> order;
    auto slot = [&](const std::vector<int32_t>& p) -> Hyp& {  // defaultdict(lambda: (-inf, -inf)) in insertion order
        const std::string k = key_of(p);
        auto it = index.find(k);
        if (it != index.end()) return next[it->second];
        index.emplace(k, (int)next.size());
        next.push_back(Hyp{p, NINF, NINF});
        return next.back();
    };
    std::vector<int32_t> ext;
    for (int t = 0; t < frames; ++t) {
        next.clear();
        index.clear();
        for (int j = 0; j < K; ++j) {
            const int s = topk_idx[(long)t * K + j];
            if (s < 0) continue;
            const double ps = (double)topk_logp[(long)t * K + j];
            // NOTE: `cur` is not modified inside this loop; `slot` may reallocate `next` only
            for (size_t h = 0; h < cur.size(); ++h) {
                const std::vector<int32_t>& prefix = cur[h].prefix;
                const double pb = cur[h].pb, pnb = cur[h].pnb;
                const bool has_last = !prefix.empty();
                if (s == blank) {
                    Hyp& e = slot(prefix);
                    const double a[3] = {e.pb, pb + ps, pnb + ps};
                    e.pb = log_add(a, 3);
                } else if (has_last && s == prefix.back()) {
                    {
                        Hyp& e = slot(prefix);  // *ss -> *s
                        const double a[2] = {e.pnb, pnb + ps};
                        e.pnb = log_add(a, 2);
                    }
                    ext = prefix;
                    ext.push_back(s);
                    Hyp& e2 = slot(ext);        // *s-s -> *ss
                    const double a2[2] = {e2.pnb, pb + ps};
                    e2.pnb = log_add(a2, 2);
                } else {
                    ext = prefix;
                    ext.push_back(s);
                    Hyp& e = slot(ext);
                    const double a[3] = {e.pnb, pb + ps, pnb + ps};
                    e.pnb = log_add(a, 3);
                }
            }
        }
        order.clear();
        for (size_t i = 0; i < next.size(); ++i) {
            const double a[2] = {next[i].pb, next[i].pnb};
            order.emplace_back(log_add(a, 2), (int)i);
        }
        std::stable_sort(order.begin(), order.end(), [](const std::pair<double, int>& x, const std::pair<double, int>& y) { return x.first > y.first; });
        const size_t keep = std::min((size_t)beam, order.size());
        std::vector<Hyp> nc;
        nc.reserve(keep);
        for (size_t i = 0; i < keep; ++i) nc.push_back(std::move(next[order[i].second]));
        cur.swap(nc);
    }
    const int n = (int)std::min((size_t)beam, cur.size());
    for (int i = 0; i < n; ++i) {
        const int len = (int)cur[i].prefix.size();
        LASR_REQUIRE(len <= max_len, "ctc_prefix_beam_search: hypothesis of %d tokens exceeds max_len %d", len, max_len);
        for (int j = 0; j < max_len; ++j) out_tokens[(long)i * max_len + j] = j < len ? cur[i].prefix[j] : -1;
        out_lens[i] = len;
        const double a[2] = {cur[i].pb, cur[i].pnb};
        out_scores[i] = log_add(a, 2);
    }
    *n_out = n;
    return LASR_OK;
}

}  // extern "C"
