// Shared helpers for the lc2is_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <atomic>

#include "../../include/lc2is_b200.h"

namespace lc2is {

// ---- error plumbing (no exception crosses the C ABI) -------------------------------------
extern thread_local char g_err[512];
extern std::atomic<long long> g_launches;

inline int fail(int code, const char* fmt, const char* a = "", long long x = 0, long long y = 0) {
    snprintf(g_err, sizeof(g_err), fmt, a, x, y);
    return code;
}
inline int cuda_fail(cudaError_t e, const char* where) {
    snprintf(g_err, sizeof(g_err), "%s: %s", where, cudaGetErrorString(e));
    return (int)e;
}
#define LC2IS_CHECK_LAUNCH(name)                                        \
    do {                                                                \
        cudaError_t e__ = cudaGetLastError();                           \
        if (e__ != cudaSuccess) return lc2is::cuda_fail(e__, name);     \
        lc2is::g_launches.fetch_add(1, std::memory_order_relaxed);      \
    } while (0)
#define LC2IS_CUDA(call)                                                \
    do {                                                                \
        cudaError_t e__ = (call);                                       \
        if (e__ != cudaSuccess) return lc2is::cuda_fail(e__, #call);    \
    } while (0)

int ensure_device();          // returns 0 or LC2IS_ERR_NODEVICE (sets g_err)
int sm_count();

inline int class_pad(int C) { return (C + 15) / 16 * 16; }

// ---- 4x4 pixel-block geometry shared by K2 and K3-lowres ---------------------------------
// For an integer power-of-two upsampling factor s >= 4 (align_corners=False), output pixels
// y in [s*j + s/2, s*(j+1) + s/2) all interpolate between source rows j and j+1.  A 4x4 pixel
// block whose origin is y0 = 4*by - off, off = (4 - (s/2)%4)%4, never straddles such a
// boundary, so its 16 pixels share one set of taps.  (torch ATen/native/UpSample.h:289-312:
// src = scale*(dst+0.5)-0.5.)
struct BlockGeom {
    int s;       // integer scale
    int off;     // pixel offset of block grid
    int nby, nbx; // number of 4x4 blocks per image in y / x
    float rs;    // 1/s
};
inline BlockGeom make_geom(int H, int W, int s) {
    BlockGeom g;
    g.s = s;
    g.off = (4 - (s / 2) % 4) % 4;
    g.nby = (H + g.off + 3) / 4;
    g.nbx = (W + g.off + 3) / 4;
    g.rs = 1.0f / (float)s;
    return g;
}
inline bool fast_scale(int h, int w, int H, int W, int* s_out) {
    if (h <= 0 || w <= 0 || H % h || W % w) return false;
    int s = H / h;
    if (W / w != s) return false;
    if (s < 4 || (s & (s - 1))) return false;
    *s_out = s;
    return true;
}

// ---- device helpers -----------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float ex2f(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcpf(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float lg2f(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// ---- interpolation weights (torch ATen/native/UpSample.h) ---------------------------------------
// bicubic: A = -0.75, src = scale*(dst+0.5)-0.5 NOT clamped, taps floor(src)-1..+2 index-clamped
// (UpSample.h:398-438, upsample_get_value_bounded).  bilinear: src clamped to >= 0
// (UpSample.h:289-312), taps idx0, min(idx0+1, in-1).
__device__ __forceinline__ float cubic1(float x, float A) { return ((A + 2.f) * x - (A + 3.f)) * x * x + 1.f; }
__device__ __forceinline__ float cubic2(float x, float A) { return ((A * x - 5.f * A) * x + 8.f * A) * x - 4.f * A; }
__device__ __forceinline__ void cubic_coeffs(float t, float (&c)[4]) {
    const float A = -0.75f;
    c[0] = cubic2(t + 1.f, A);
    c[1] = cubic1(t, A);
    c[2] = cubic1(1.f - t, A);
    c[3] = cubic2(2.f - t, A);
}
__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// ---- programmatic dependent launch ---------------------------------------------------------------
// A kernel started by launch_pdl may begin while the kernel before it on the stream is still running: everything up to
// griddep_wait() (barrier init, TMEM allocation, tensor-map prefetch, loads of inputs older than the predecessor) overlaps
// that kernel's tail.  griddep_wait() returns once the predecessor has COMPLETED and its writes are visible, so every
// thread of such a kernel must pass it before it reads the predecessor's output or writes anything the predecessor reads;
// a kernel that does not call it could finish before its predecessor, breaking the transitive order of a chain.
// griddep_launch_dependents() lets the next kernel of the stream be scheduled once every CTA has issued it (or exited).
// Without a programmatic predecessor (a memset, an event wait, a plain launch) both are no-ops.
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args&&... args) {
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}


}  // namespace lc2is
