// runtime.cu -- library-level services of libhpc_rll_b200.so: error text, launch counter,
// TMA descriptor encoding through the driver entry point, tuning overrides.
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "common.cuh"

namespace hpcrll {

static thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};
static std::atomic<int> g_cfg[HPC_RLL_OP_COUNT];
static std::once_flag g_cfg_once;

int set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
void clear_error() { g_err[0] = '\0'; }
void count_launch(int n) { g_launches.fetch_add(static_cast<uint64_t>(n), std::memory_order_relaxed); }

int sm_count() {
    static thread_local int cached_dev = -1, cached = 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (dev != cached_dev) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached = n;
        cached_dev = dev;
    }
    return cached;
}

static void init_cfg() {
    static const char* names[HPC_RLL_OP_COUNT] = {"GAE", "TD_LAMBDA", "VTRACE", "UPGO", "PPO",
                                                  "Q_NSTEP_TD", "DIST_NSTEP_TD", "QRDQN_NSTEP_TD", "IQN_NSTEP_TD",
                                                  "GAE_MOMENTS", "SCATTER_CONNECTION"};
    for (int i = 0; i < HPC_RLL_OP_COUNT; ++i) {
        char key[64];
        snprintf(key, sizeof(key), "HPC_RLL_CFG_%s", names[i]);
        const char* v = getenv(key);
        g_cfg[i].store(v ? atoi(v) : -1);
    }
}
int tuning_config(int op) {
    std::call_once(g_cfg_once, init_cfg);
    if (op < 0 || op >= HPC_RLL_OP_COUNT) return -1;
    return g_cfg[op].load();
}

// ---- TMA descriptor encode -------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    });
    return fn;
}

bool tma_ok_2d(const void* base, int64_t cols, int64_t ld) {
    return aligned16(base) && cols > 0 && ld >= cols && (ld % 4) == 0 && ld < (int64_t(1) << 38);
}

int make_tmap_2d(CUtensorMap* out, const float* base, int64_t rows, int64_t cols, int64_t ld, int box_rows,
                 int box_cols, bool swizzle128) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return set_error(HPC_RLL_ECUDA, "cuTensorMapEncodeTiled entry point unavailable");
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * sizeof(float)};
    cuuint32_t box[2] = {static_cast<cuuint32_t>(box_cols), static_cast<cuuint32_t>(box_rows)};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return set_error(HPC_RLL_ECUDA, "cuTensorMapEncodeTiled failed (%d) rows=%lld cols=%lld ld=%lld", (int)r,
                         (long long)rows, (long long)cols, (long long)ld);
    return HPC_RLL_OK;
}

}  // namespace hpcrll

extern "C" {

const char* hpc_rll_version(void) { return "hpc_rll_b200 0.1 (sm_100a)"; }
const char* hpc_rll_last_error(void) { return hpcrll::g_err; }
uint64_t hpc_rll_launch_count(void) { return hpcrll::g_launches.load(); }

size_t hpc_rll_workspace_bytes(int op, int64_t T, int64_t B, int64_t N) {
    return hpcrll::workspace_bytes(op, T, B, N);
}

int hpc_rll_debug_set_config(int op, int cfg) {
    hpcrll::tuning_config(0);  // make sure env defaults were read first
    if (op < 0 || op >= HPC_RLL_OP_COUNT) return hpcrll::set_error(HPC_RLL_EINVAL, "bad op id %d", op);
    hpcrll::g_cfg[op].store(cfg);
    return HPC_RLL_OK;
}

}  // extern "C"
