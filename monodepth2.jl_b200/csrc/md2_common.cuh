// Host-side plumbing shared by the .cu translation units: context, error reporting,
// workspace, launch accounting, block reductions.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <stdio.h>

#include "../../include/md2.h"
#include "md2_math.cuh"

namespace md2 {

std::string& last_error_ref();
int set_error(const char* fmt, ...);

struct Workspace {
    void* ptr = nullptr;
    size_t bytes = 0;
};

}  // namespace md2

enum { MD2_WS_PARTIAL = 0, MD2_WS_SUMS, MD2_WS_POSE, MD2_WS_STATS, MD2_WS_DISP, MD2_WS_GDISP,
       MD2_WS_MISC, MD2_WS_AUTOMASK, MD2_WS_KGRAD, MD2_WS_COUNT };
// workspace banks: calls that may be in flight at the same time must not share scratch.  Bank 0 serves the
// device-pointer entry points (one stream at a time, md2.h), banks 1.. the lanes of the host-buffer entry point.
enum { MD2_WS_BANKS = 1 + MD2_HOST_LANES };

#include <vector>
struct md2_ctx {
    int device;
    int64_t launches;
    int sm_count = 148;
    int bank = 0;                          // workspace bank the next run_vsl uses (set by the entry points)
    int64_t ws_gen[MD2_WS_BANKS] = {};     // bumped whenever a slot of the bank is (re)allocated: captured CUDA graphs hold the old pointers
    md2::Workspace ws[MD2_WS_BANKS][MD2_WS_COUNT];
    // optional device timing of the dominant (fused tile) kernel, see md2_profile_*
    int prof_on = 0;
    std::vector<cudaEvent_t> prof_ev;   // start/stop pairs
    size_t prof_used = 0;
    void* host[MD2_HOST_LANES] = {};   // lanes of the host-buffer entry point (md2_host.cu), created on first use
    void* opt = nullptr;    // state of md2_slow_depth (md2_optim.cu), created on first use
    void* taps = nullptr;   // upsample tap tables per shape (md2_fused.cu), created on first use
    void* replay = nullptr; // CUDA-graph cache of the device-pointer fused calls (md2_fused.cu), created on first use
};

namespace md2 {

// returns nullptr (and sets the error) on failure
void* ws_get(md2_ctx* ctx, int slot, size_t bytes);
// md2_ops.cu: out (N,1,H,W) = min over the S frames of photometric_loss(frame_s, target) (automasking_loss on frame views)
int launch_automask(md2_ctx* ctx, int S, const float* const* frames, const int64_t* frame_ns, const float* target, int64_t target_ns,
                    float* out, int W, int H, int C, int N, cudaStream_t st);

// the C entry points make the ctx's device current for the duration of the call and restore the caller's device
struct DeviceGuard {
    int prev = -1;
    cudaError_t err;
    explicit DeviceGuard(int device) {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != device) err = cudaSetDevice(device); else if (err == cudaSuccess) prev = -1;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
#define MD2_USE_DEVICE(ctx)                \
    md2::DeviceGuard _dev_guard((ctx)->device); \
    MD2_CHECK(_dev_guard.err)

#define MD2_CHECK(expr)                                                                  \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess)                                                           \
            return md2::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                                  __FILE__, __LINE__);                                   \
    } while (0)

#define MD2_LAUNCH_CHECK(ctx)                                                           \
    do {                                                                                \
        (ctx)->launches++;                                                              \
        cudaError_t _e = cudaGetLastError();                                            \
        if (_e != cudaSuccess)                                                          \
            return md2::set_error("kernel launch failed: %s (%s:%d)",                   \
                                  cudaGetErrorString(_e), __FILE__, __LINE__);          \
    } while (0)

#define MD2_REQUIRE(cond, msg)                                  \
    do {                                                        \
        if (!(cond)) return md2::set_error("%s: %s", __func__, msg); \
    } while (0)

#if defined(__CUDACC__)
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Warp-aggregated scatter of one bilinear tap pair (left tap aL += vL, right tap aR += vR; nullptr = the tap does not exist).
// Neighbouring lanes hold neighbouring output pixels, and under a smooth warp lane i's RIGHT tap is the very address of
// lane i+1's LEFT tap: the pair is merged in registers (one shuffle each way) and issued as ONE red.global.add by the
// receiving lane, so a pixel costs ~1 atomic per tap row and channel instead of 2 (the per-tap atomicAdd of a
// thread-per-pixel sampler backward -- NNlib's -- serialises exactly those collisions in the L2).
// Must be called by all 32 lanes of the warp (lanes without work pass nullptrs).
__device__ __forceinline__ void red_pair_merged(float* aL, float* aR, float vL, float vR, int lane) {
    const unsigned long long nbL = __shfl_down_sync(0xffffffffu, reinterpret_cast<unsigned long long>(aL), 1);
    const bool give = aR != nullptr && lane < 31 && nbL == reinterpret_cast<unsigned long long>(aR);
    const float recv = __shfl_up_sync(0xffffffffu, give ? vR : 0.f, 1);
    if (aL) atomicAdd(aL, lane > 0 ? vL + recv : vL);
    if (aR && !give) atomicAdd(aR, vR);
}

// Deterministic block-wide sum of NV values per thread; result valid in thread 0's out[].
// scratch must hold NV * (blockDim.x/32) floats.
template <int NV>
__device__ __forceinline__ void block_sum(float (&v)[NV], float* scratch) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        const float s = warp_sum(v[k]);
        if (lane == 0) scratch[k * nw + wid] = s;
    }
    __syncthreads();
    if (threadIdx.x < NV) {
        float s = 0.f;
        for (int w = 0; w < nw; ++w) s += scratch[threadIdx.x * nw + w];
        scratch[threadIdx.x * nw] = s;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < NV; ++k) v[k] = scratch[k * nw];
    __syncthreads();
}

// Julia column-major 3x3 -> row-major doubles
__device__ __forceinline__ void load_cm3(const float* m, double* o) {
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) o[3 * i + j] = (double)m[3 * j + i];
}
#endif

inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

}  // namespace md2
