// Host-side helpers shared by the C-ABI entry points: error string, launch counter, TMA descriptor encoding.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>
#include <functional>

namespace omg {

extern thread_local char g_err[512];
extern std::atomic<uint64_t> g_launches;

inline int fail(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return 1;
}

#define OMG_CHECK(cond, ...) \
    do {                     \
        if (!(cond)) return ::omg::fail(__VA_ARGS__); \
    } while (0)

#define OMG_CUDA(expr)                                                                       \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) return ::omg::fail("%s failed: %s", #expr, cudaGetErrorString(_e)); \
    } while (0)

inline int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail("launch of %s failed: %s", what, cudaGetErrorString(e));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

// Launch plans (omg_plan_*, include/omg_b200.h): while a thread records, every entry point that launched successfully also
// appends a replayable copy of its call (descriptors by value) to the plan; omg_plan_run re-issues them on a stream.
bool plan_recording();
void plan_note(std::function<int(void*)> step);

// Every kernel of this library can be launched with programmatic dependent launch (PDL): the next kernel's CTAs may
// become resident and run their prologue (barrier init, TMEM alloc, descriptor prefetch) while the previous kernel
// drains; each kernel executes griddepcontrol.wait before its first dependent global access.  Measured on the full
// two-stage loop inside CUDA graphs: 2791.8 ms/image with the attribute, 2770.4 ms without (no gain: the one-CTA-per-
// SM kernels cannot co-reside anyway), so it is opt-in: OMG_PDL=1.
bool pdl_enabled();

template <typename... KArgs, typename... Args>
inline cudaError_t launch_cluster(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                  int cluster_x, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    int n = 0;
    if (pdl_enabled()) {
        attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[n].val.programmaticStreamSerializationAllowed = 1;
        ++n;
    }
    if (cluster_x > 1) {
        attr[n].id = cudaLaunchAttributeClusterDimension;
        attr[n].val.clusterDim.x = cluster_x;
        attr[n].val.clusterDim.y = 1;
        attr[n].val.clusterDim.z = 1;
        ++n;
    }
    cfg.attrs = attr;
    cfg.numAttrs = n;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              Args... args) {
    return launch_cluster(kernel, grid, block, smem, stream, 1, args...);
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// libcuda is resolved at run time through the runtime (the build box has no driver library to link against).
PFN_encodeTiled get_encode_tiled();

// Tensor map of 16-bit elements (`dtype` FLOAT16 or BFLOAT16) of rank `rank` (<=5). dims[0] is the contiguous dimension.
// strides are in ELEMENTS for dims[1..rank-1].  Out-of-bounds box elements read as zero / are clipped on store.
int make_tmap_16b(CUtensorMap* out, const void* ptr, int rank, const uint64_t* dims, const uint64_t* strides_elems,
                  const uint32_t* box, CUtensorMapSwizzle swizzle,
                  CUtensorMapDataType dtype = CU_TENSOR_MAP_DATA_TYPE_FLOAT16);

}  // namespace omg
