// Internal helpers shared by the .cu translation units of libadm_b200.so.
#pragma once
#include <stdarg.h>
#include <cuda.h>
#include <cuda_runtime.h>
#include "../../include/adm_b200.h"

namespace adm {
void set_error(const char* fmt, ...);
const char* get_error();
int num_sms();
void count_launch();
// bf16 tensor map, 128B swizzle, zero OOB fill.  dims/box innermost first; strides in ELEMENTS for dims 1..rank-1.
// Returns 0, or ADM_ERR_SHAPE / ADM_ERR_CUDA with the error set.
int encode_map(CUtensorMap* m, const void* ptr, int rank, const long long* dims, const long long* strides,
               const int* box);

#ifdef __CUDACC__
// <<<>>> replacement for the hot kernels: optional thread-block cluster.
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s,
                                   int cluster_x, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    if (cluster_x > 0) {
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = cluster_x;
        at[0].val.clusterDim.y = 1;
        at[0].val.clusterDim.z = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
    }
    return cudaLaunchKernelEx(&cfg, kern, args...);
}

// Raises Kern's dynamic shared-memory limit to `bytes` on the first successful call.  The flag is keyed on the kernel
// itself, not on its signature: the GEMM engine's kernels all share one parameter list.
template <auto Kern>
static inline cudaError_t set_smem_limit_once(int bytes) {
    static bool done = false;
    if (done) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    done = e == cudaSuccess;
    return e;
}
#endif

#define ADM_CHECK_LAUNCH(name)                                              \
    do {                                                                    \
        cudaError_t e__ = cudaGetLastError();                               \
        if (e__ != cudaSuccess) {                                           \
            adm::set_error("%s launch: %s", name, cudaGetErrorString(e__)); \
            return ADM_ERR_CUDA;                                            \
        }                                                                   \
        adm::count_launch();                                                \
    } while (0)
}  // namespace adm
