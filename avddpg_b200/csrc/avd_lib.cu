// avd_lib.cu -- library-level entry points: ABI version, last-error text, device probe; the tensor-map encoder.
#include <cudaTypedefs.h>
#include <cstdlib>
#include <stdarg.h>
#include <string.h>

#include <atomic>

#include "avd_common.cuh"
#include "avd_umma.cuh"

namespace avd {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

static std::atomic<long long> g_launches{0};

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

bool pdl_enabled() {
    static const bool on = [] {
        const char* e = getenv("AVD_PDL");
        return !(e && e[0] == '0');
    }();
    return on;
}

int sm_count() {
    static int cached = 0;
    if (cached == 0) {
        int dev = 0, n = 0;
        if (cudaGetDevice(&dev) == cudaSuccess &&
            cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
            cached = n;
        else
            return 148;  // B200; only reached when no device is visible (launches then fail loudly)
    }
    return cached;
}

int umma::make_tensor_map(CUtensorMap* map, const void* base, uint64_t inner, uint64_t rows, uint64_t batch, uint64_t pitch,
                          uint64_t batch_stride, uint32_t box_inner, uint32_t box_rows) {
    static PFN_cuTensorMapEncodeTiled enc = nullptr;
    if (!enc) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            enc = reinterpret_cast<PFN_cuTensorMapEncodeTiled>(p);
    }
    if (!enc) {
        set_error("cuTensorMapEncodeTiled is not available from the driver");
        return AVD_ERR_CUDA;
    }
    cuuint64_t dims[3] = {inner, rows, batch};
    cuuint64_t strides[2] = {pitch * 2, batch_stride * 2};
    if (batch == 1 && strides[1] == 0) strides[1] = pitch * 2 * rows;
    cuuint32_t box[3] = {box_inner, box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with %d (inner=%llu rows=%llu batch=%llu pitch=%llu)", (int)r, (unsigned long long)inner,
                  (unsigned long long)rows, (unsigned long long)batch, (unsigned long long)pitch);
        return AVD_ERR_CUDA;
    }
    return AVD_OK;
}

}  // namespace avd

extern "C" int avd_abi_version(void) { return AVD_ABI_VERSION; }

extern "C" const char* avd_last_error(void) { return avd::g_err; }

extern "C" int64_t avd_kernel_launches(void) { return (int64_t)avd::g_launches.load(std::memory_order_relaxed); }

extern "C" int64_t avd_sizeof(int which) {
    switch (which) {
        case 0: return (int64_t)sizeof(avd_env_params);
        case 1: return (int64_t)sizeof(avd_env_io);
        case 2: return (int64_t)sizeof(avd_clock);
        case 3: return (int64_t)sizeof(avd_net_dims);
        case 4: return (int64_t)sizeof(avd_learn_io);
        case 5: return (int64_t)sizeof(avd_peer_comm);
        case 6: return (int64_t)sizeof(avd_fed_apply_io);
        case 7: return (int64_t)sizeof(avd_runs);
        default: return -1;
    }
}

extern "C" int avd_device_info(int* sm_count_out, int* cc, int64_t* total_mem) {
    int dev = 0;
    cudaDeviceProp prop;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&prop, dev) != cudaSuccess) {
        cudaGetLastError();
        avd::set_error("no CUDA device visible: libavddpg_b200 has no CPU fallback");
        return AVD_ERR_NO_DEVICE;
    }
    if (sm_count_out) *sm_count_out = prop.multiProcessorCount;
    if (cc) *cc = prop.major * 10 + prop.minor;
    if (total_mem) *total_mem = (int64_t)prop.totalGlobalMem;
    if (prop.major != 10) {
        avd::set_error("device is sm_%d%d; this library is compiled for sm_100a only", prop.major, prop.minor);
        return AVD_ERR_NO_DEVICE;
    }
    return AVD_OK;
}
