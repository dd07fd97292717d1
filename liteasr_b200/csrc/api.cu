// C-ABI glue: error reporting, version, and the GEMM dispatcher.
#include <cstdarg>
#include <cstdio>

#include "common.cuh"

namespace lasr {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

static unsigned long long g_launches = 0;

int check_launch(const char* what) {
    ++g_launches;  // one per kernel launch site (statistics only; benign race across threads)
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return LASR_ERR_CUDA;
    }
    return LASR_OK;
}

int gemm_tc_dispatch(const lasr_gemm_args* a, cudaStream_t st);
int gemm_simt_dispatch(const lasr_gemm_args* a, cudaStream_t st);

}  // namespace lasr

extern "C" {

int lasr_version(void) { return 2; }
int lasr_arch(void) { return 100; }
const char* lasr_last_error(void) { return lasr::g_err; }
unsigned long long lasr_launch_count(void) { return lasr::g_launches; }

int lasr_gemm(const lasr_gemm_args* a, void* stream) {
    using namespace lasr;
    LASR_REQUIRE(a && a->a && a->b && a->c, "gemm: null operand");
    LASR_REQUIRE(a->m > 0 && a->n > 0 && a->k > 0, "gemm: bad shape m=%d n=%d k=%d", a->m, a->n, a->k);
    LASR_REQUIRE(a->batch1 >= 1 && a->batch2 >= 1, "gemm: bad batch");
    LASR_REQUIRE((long)a->batch1 * a->batch2 * (a->split_k < 1 ? 1 : a->split_k) <= 65535, "gemm: batch*split_k > 65535");
    if (a->accumulate)
        LASR_REQUIRE(a->c_dtype == LASR_F32 && !a->bias && !a->res && !a->aux && !a->dact && !a->colsum && a->act == LASR_ACT_NONE,
                     "gemm: accumulate needs fp32 C and no epilogue");
    if (a->dact)
        LASR_REQUIRE(!a->bias && !a->res && !a->aux && (a->act == LASR_ACT_SWISH || a->act == LASR_ACT_RELU || a->act == LASR_ACT_MUL) && a->lddact > 0,
                     "gemm: dact needs act = swish|relu|mul and no bias/res/aux");
    else
        LASR_REQUIRE(a->act != LASR_ACT_MUL, "gemm: act = mul needs dact");
    if (a->aux_deriv) LASR_REQUIRE(a->aux && a->act == LASR_ACT_SWISH, "gemm: aux_deriv needs aux and act = swish");
    if (a->split_k > 1) LASR_REQUIRE(a->accumulate, "gemm: split_k > 1 requires accumulate");
    if (a->n_store)
        LASR_REQUIRE(a->n_store >= a->n && a->n_store <= a->ldc && !a->bias && !a->res && !a->aux && !a->dact && !a->colsum && !a->accumulate,
                     "gemm: n_store must satisfy n <= n_store <= ldc and excludes every epilogue operand");
    if (a->drop_thr)
        LASR_REQUIRE(a->drop_state && a->drop_thr <= 0x7c00u && a->batch1 == 1 && a->batch2 == 1 && !a->accumulate && !a->dact && !a->n_store &&
                         !a->colsum,
                     "gemm: dropout needs drop_state, thr = round(p * 32768) <= 0x7c00, an unbatched GEMM and no accumulate / dact / n_store / colsum");
    cudaStream_t st = (cudaStream_t)stream;
    if (a->ab_dtype == LASR_BF16) return gemm_tc_dispatch(a, st);
    if (a->ab_dtype == LASR_F32) {
        LASR_REQUIRE(a->c_dtype == LASR_F32, "gemm: fp32 operands need fp32 C");
        return gemm_simt_dispatch(a, st);
    }
    set_error("gemm: unsupported dtype %d", a->ab_dtype);
    return LASR_ERR_UNSUPPORTED;
}

}  // extern "C"
