// Shared host/device helpers of libmugd (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <utility>

#include "../../include/mugd.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libmugd is written for sm_100a (B200) only"
#endif

namespace mugd {

void set_error(const char* fmt, ...);

#define MUGD_CHECK_CUDA(expr)                                                             \
    do {                                                                                  \
        cudaError_t _e = (expr);                                                          \
        if (_e != cudaSuccess) {                                                          \
            ::mugd::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr,                \
                              cudaGetErrorString(_e));                                    \
            return MUGD_ERR_CUDA;                                                         \
        }                                                                                 \
    } while (0)

#define MUGD_REQUIRE(cond, ...)                                                           \
    do {                                                                                  \
        if (!(cond)) {                                                                    \
            ::mugd::set_error(__VA_ARGS__);                                               \
            return MUGD_ERR_INVALID;                                                      \
        }                                                                                 \
    } while (0)

struct DeviceInfo {
    int device = 0;
    int sm_count = 148;
    int cc_major = 0, cc_minor = 0;
    int max_smem_optin = 0;
    // per-handle switches (round 1 kept these as process globals)
    int tc_single_pass = 0;     // opt-in plain-TF32 tensor-core products (NOT fp32-accurate; never used by parity tests / bench)
    int attention_impl = 1;     // 1 = tcgen05 attention, 0 = exact-fp32 FFMA referee
};

// per-family launchers (each validates its descriptor and enqueues kernels on `st`);
// they return the number of kernels launched through *launches (may be null)
int launch_gemm(const DeviceInfo& dev, const mugd_gemm& g, int default_impl, cudaStream_t st, int* launches);
int launch_groupnorm(const DeviceInfo& dev, const mugd_groupnorm& g, cudaStream_t st, int* launches);
int launch_layernorm(const DeviceInfo& dev, const mugd_layernorm& g, cudaStream_t st, int* launches);
int launch_attention(const DeviceInfo& dev, const mugd_attention& a, cudaStream_t st, int* launches);
int launch_s4conv(const DeviceInfo& dev, const mugd_s4conv& s, cudaStream_t st, int* launches);
int launch_ddim_update(const DeviceInfo& dev, const mugd_ddim_update& d, cudaStream_t st, int* launches);
int launch_transpose(const DeviceInfo& dev, const mugd_transpose& t, cudaStream_t st, int* launches);
int launch_copy2d(const DeviceInfo& dev, const mugd_copy2d& c, cudaStream_t st, int* launches);
int launch_step_advance(const DeviceInfo& dev, const mugd_step_advance& a, cudaStream_t st, int* launches);
int launch_notes(const DeviceInfo& dev, const mugd_notes& n, cudaStream_t st, int* launches);
int launch_embed(const DeviceInfo& dev, const mugd_embed& e, cudaStream_t st, int* launches);
int launch_tf32_split(const DeviceInfo& dev, const mugd_tf32_split& s, cudaStream_t st, int* launches);
int launch_gemm_tc(const DeviceInfo& dev, const mugd_gemm& g, cudaStream_t st, int* launches);
bool gemm_tc_supported(const mugd_gemm& g);

// Kernel attributes are per device: mugd_create sets them on its device for every instantiation the launchers can pick (dynamic
// shared memory above the 48 KB default, carveout).
int configure_gemm_tc_kernels(const DeviceInfo& dev);
int configure_attention_kernels(const DeviceInfo& dev);
int configure_attention_tc_kernels(const DeviceInfo& dev);
int configure_s4_kernels(const DeviceInfo& dev);

// Programmatic dependent launch (PDL): launch_k always sets the programmatic-stream-serialization attribute, and every kernel it
// launches executes `griddepcontrol.wait` before its first global-memory access.  The next kernel's launch latency and prologue
// (block scheduling, barrier init, TMEM allocation, tensor-map fetch) then overlap the tail of the current one; data hazards
// are unchanged because the wait only returns when the prerequisite grid has completed and flushed.

#ifdef __CUDACC__
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}
// No kernel signals launch_dependents explicitly: the trigger is implicit at grid completion, so PDL only overlaps the dependent's
// launch with this grid's memory flush (graph edge 0.57 us instead of 0.69 us, tools/experiments/sync_probe.cu).  Explicit triggers
// (at entry, in the short kernels only, after the GEMM main loop) were measured slower in round 1 (DESIGN.md 4) and removed.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---- device helpers ---------------------------------------------------------------------------
__device__ __forceinline__ float silu_f(float x) { return x / (1.0f + expf(-x)); }
__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + expf(-x)); }
// exact-erf GELU (nn.GELU() default; attention.py:45, s4.py:187-188)
__device__ __forceinline__ float gelu_f(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }

__device__ __forceinline__ float4 ld_f4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st_f4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
#endif

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// cuTensorMapEncodeTiled of the driver the runtime runs on (tensor maps of the tcgen05 GEMM and attention); null if unavailable
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) == cudaSuccess && qr == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

}  // namespace mugd
