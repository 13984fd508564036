// Fused view-synthesis loss: __global__ wrappers around md2_fused.cuh + host orchestration
// + the C ABI (md2_view_synthesis_loss_{fwd,bwd,fwdbwd}).  sm_100a only.
#include <stdarg.h>
#include <string.h>

#include <atomic>

#include "md2_common.cuh"
#include "md2_fused.cuh"
#include "md2_march.cuh"
#include "md2_march2.cuh"

namespace md2 {

void host_path_destroy(md2_ctx* ctx);   // md2_host.cu
void opt_path_destroy(md2_ctx* ctx);    // md2_optim.cu
void replay_destroy(md2_ctx* ctx);
void taps_destroy(md2_ctx* ctx);

// ------------------------------------------------------------------------------------------
// error / ctx plumbing
// ------------------------------------------------------------------------------------------
std::string& last_error_ref() {
    static thread_local std::string e;
    return e;
}
int set_error(const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    last_error_ref() = buf;
    return 1;
}
void* ws_get(md2_ctx* ctx, int slot, size_t bytes) {
    Workspace& w = ctx->ws[ctx->bank][slot];
    if (w.bytes >= bytes && w.ptr) return w.ptr;
    if (w.ptr) {
        cudaDeviceSynchronize();  // growth only: a previous launch may still read the old buffer
        cudaFree(w.ptr);
        w.ptr = nullptr; w.bytes = 0;
    }
    size_t want = bytes + bytes / 4 + 256;
    ctx->ws_gen[ctx->bank]++;
    cudaError_t e = cudaMalloc(&w.ptr, want);
    if (e != cudaSuccess) {
        set_error("workspace cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
        w.ptr = nullptr;
        return nullptr;
    }
    w.bytes = want;
    return w.ptr;
}

// ------------------------------------------------------------------------------------------
// align-corners bilinear upsample (A17) and its adjoint as stand-alone operators
// ------------------------------------------------------------------------------------------
__global__ void upsample_kernel(const float* __restrict__ in, float* __restrict__ out, int w, int h,
                                int W, int H, int CN) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)W * H * CN) return;
    const int x = (int)(i % W), y = (int)((i / W) % H);
    const long long cn = i / ((long long)W * H);
    const float sx = up_scale(w, W), sy = up_scale(h, H);
    int x0, x1, y0, y1; float fx, fy;
    up_taps(x, w, W, x0, x1, fx);
    up_taps(y, h, H, y0, y1, fy);
    const float* b = in + cn * w * h;
    out[i] = bilerp(b[y0 * w + x0], b[y0 * w + x1], b[y1 * w + x0], b[y1 * w + x1], fx, fy);
}

// gather form (deterministic): one thread per low-resolution pixel
__global__ void upsample_bwd_kernel(const float* __restrict__ gout, float* __restrict__ gin, int w,
                                    int h, int W, int H, int CN) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)w * h * CN) return;
    const int xi = (int)(i % w), yi = (int)((i / w) % h);
    const long long cn = i / ((long long)w * h);
    gin[i] = upsample_adjoint_at(gout + cn * W * H, w, h, W, H, xi, yi);
}

// out[g][k] = sum_b partial[g][b][k], fixed order (deterministic).  NP <= 32.
// Columns k < n0 go to out0 (row length n0), the rest to out1 (row length NP - n0).
__global__ void __launch_bounds__(256) reduce_partials_kernel(const float* __restrict__ partial,
                                                              float* __restrict__ out0, int n0,
                                                              float* __restrict__ out1, int bpg, int NP) {
    __shared__ float sm[8][32];
    const int g = blockIdx.x, k = threadIdx.x & 31, chunk = threadIdx.x >> 5;
    float s = 0.f;
    if (k < NP)
        for (int b = chunk; b < bpg; b += 8) s += partial[((long long)g * bpg + b) * NP + k];
    sm[chunk][k] = s;
    __syncthreads();
    if (chunk == 0 && k < NP) {
        float t = 0.f;
        for (int c = 0; c < 8; ++c) t += sm[c][k];
        if (k < n0) out0[(long long)g * n0 + k] = t;
        else if (out1) out1[(long long)g * (NP - n0) + (k - n0)] = t;
    }
}

int launch_reduce_partials(md2_ctx* ctx, const float* partial, float* out0, int n0, float* out1,
                           int groups, int bpg, int NP, cudaStream_t st) {
    reduce_partials_kernel<<<groups, 256, 0, st>>>(partial, out0, n0, out1, bpg, NP);
    MD2_LAUNCH_CHECK(ctx);
    return 0;
}

// ------------------------------------------------------------------------------------------
// programmatic dependent launch: with MD2_PDL (bit mask, see pdl_mask) the three kernels of a call are chained with
// cudaLaunchAttributeProgrammaticStreamSerialization, so the next kernel's blocks are scheduled (launch latency, block
// set-up) while the previous kernel drains; pdl_wait() returns once the previous kernel has completed and its writes are
// visible, pdl_trigger() lets the next kernel start launching.  Default 0 = plain stream order: measured faster (the
// dependent's early-resident warps take registers from the running kernel: 83.0 vs 74.6 us per step at 416x128x8).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
#ifndef MD2_PDL_EARLY
#define MD2_PDL_EARLY 1   // 1: a block lets the dependent kernel start launching as soon as it runs; 0: only when it exits
#endif
__device__ __forceinline__ void pdl_trigger() {
#if MD2_PDL_EARLY
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
}

// bit 0: the marching kernel may overlap the prep kernel's tail, bit 1: the finish kernel the marching kernel's
static int pdl_mask() {
    static const int m = [] { const char* e = getenv("MD2_PDL"); return e ? atoi(e) : 0; }();
    return m;
}
template <class... KArgs, class... Args>
static cudaError_t launch_after(int pdl_bit, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = (pdl_mask() & pdl_bit) ? 1 : 0;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// ------------------------------------------------------------------------------------------
// warp-level helpers
// ------------------------------------------------------------------------------------------
// Transpose-reduce: every lane passes 32 values; afterwards lane k holds the warp total of
// value k.  31 shuffles instead of 32 x 5.
__device__ __forceinline__ float warp_reduce_32(float (&v)[32]) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int half = 16; half >= 1; half >>= 1) {
        const bool up = (lane & half) != 0;
#pragma unroll
        for (int i = 0; i < half; ++i) {
            const float send = up ? v[i] : v[i + half];
            const float keep = up ? v[i + half] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, half);
        }
    }
    return v[0];
}

// ------------------------------------------------------------------------------------------
// prep kernel (one launch before the marching kernel), grid (1 + nblk + S * zero_blocks, N):
//   blockIdx.x == 0 : [composeT +] pose pre-composition of image blockIdx.y (scheduled first, so
//       the serial double-precision pose maths overlaps the rest of the grid)
//   1 <= blockIdx.x <= nblk : eight warps, each owning a 31-column x 4-row patch of image
//       blockIdx.y (lane = column, lane 31 = right-hand halo; one extra row below as lower
//       neighbour), for all decoder scales.  Rows are unrolled and the loads of a scale are issued
//       up front.  (a) writes the align-corners bilinear upsample (A17) of every low-res
//       disparity into its full-resolution scratch -- separable: the (at most 4) low-res rows a
//       patch touches are interpolated horizontally once per lane, the vertical weights are
//       warp-uniform -- and (b) for the fused fwd+bwd call accumulates the smoothness /
//       mean-disparity sums of every scale (needed before the backward because d / mean(d) couples
//       all pixels of an image, SURVEY.md appendix A.6; the edge weights exp(-|dT|) are computed
//       once and shared by the scales).  Right neighbours come from the next lane, lower
//       neighbours from the next row, so every disparity is interpolated once.  One partial
//       (Sx, Sy, sum d) per block and scale; the consumers (warp B of the marching kernel, the
//       finish kernel) add the partials of a (scale, image) in a fixed order (deterministic).
//   blockIdx.x > nblk : zero-fill of one slice of a grad_source image (desc.zero_grad_source)
// ------------------------------------------------------------------------------------------
constexpr int PREP_COLS = 31;
constexpr int PREP_ROWS = 4;
constexpr int PREP_WARPS = 8;
#ifndef MD2_PREP_MINB
#define MD2_PREP_MINB 4   // resident blocks per SM the lean prep kernel is compiled for (4: 64 registers, one wave at 416x128x8, some spills)
#endif

// one entry of a tap table (FusedParams::tap_x / tap_y): the two source indices and the weight of the second
__device__ __forceinline__ void tap_load(const float* __restrict__ tab, int i, int& i0, int& i1, float& f) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(tab) + i);
    i0 = __float_as_int(t.x); i1 = __float_as_int(t.y); f = t.z;
}

__device__ __forceinline__ float sel4(const float (&h)[4], int k) {   // k is warp-uniform
    return k == 0 ? h[0] : (k == 1 ? h[1] : (k == 2 ? h[2] : h[3]));
}

// block 0 of an image: poses; blocks beyond the patch blocks: one slice of a source image each -- pull it into the L2
// (the marching kernel's gathers are the only reads of the source frames: without this they are cold DRAM misses with
// ~1000 cycles of latency in the middle of its software pipeline), and zero-fill the same slice of the source-gradient
// image when the call asks for it (zero_blocks < 0: prefetch only)
template <int C>
__device__ __forceinline__ void prep_pose_or_zero(const FusedParams& p, int nblk, float* __restrict__ pose_ab, int zero_blocks) {
    const int n = blockIdx.y;
    if (blockIdx.x == 0) {
        if ((int)threadIdx.x < p.S)
            prepare_pose_one(p.pose, threadIdx.x, n, pose_ab + ((long long)threadIdx.x * p.N + n) * 12,
                             pose_ab + ((long long)(p.S + threadIdx.x) * p.N + n) * 12);   // (the displacement table follows the A | b table)
        return;
    }
    const bool do_zero = zero_blocks > 0;
    zero_blocks = zero_blocks < 0 ? -zero_blocks : zero_blocks;
    const int zb = blockIdx.x - nblk - 1, s = zb / zero_blocks, sl = zb - s * zero_blocks;
    const int total = C * p.W * p.H;
    const int per = ((total + zero_blocks - 1) / zero_blocks + 3) & ~3;
    const int i0 = sl * per, i1 = min(i0 + per, total);
    {   // one 128-byte line per thread
        const float* src = p.src[s] + (long long)n * p.src_ns[s];
        for (int i = i0 + 32 * (int)threadIdx.x; i < i1; i += 32 * (int)blockDim.x)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(src + i));
        if (threadIdx.x == 0 && i1 > i0) asm volatile("prefetch.global.L2 [%0];" ::"l"(src + (i1 - 1)));
    }
    if (!do_zero || !p.gsrc[s]) return;
    float* g = p.gsrc[s] + (long long)n * p.src_ns[s];
    if ((reinterpret_cast<uintptr_t>(g) & 15) == 0) {
        for (int i = i0 + 4 * (int)threadIdx.x; i + 3 < i1; i += 4 * (int)blockDim.x) *reinterpret_cast<float4*>(g + i) = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int i = i0 + ((i1 - i0) & ~3) + (int)threadIdx.x; i < i1; i += blockDim.x) g[i] = 0.f;
    } else {
        for (int i = i0 + (int)threadIdx.x; i < i1; i += blockDim.x) g[i] = 0.f;
    }
}

template <int C, int LMAX>
__global__ void __launch_bounds__(32 * PREP_WARPS, 3) prep_kernel(const __grid_constant__ FusedParams p, int strips, int chunks,
                                                               int nblk, int do_stats, float* __restrict__ pose_ab,
                                                               float* __restrict__ part, int zero_blocks) {
    const int n = blockIdx.y;
    pdl_trigger();
    if (blockIdx.x == 0 || (int)blockIdx.x > nblk) { prep_pose_or_zero<C>(p, nblk, pose_ab, zero_blocks); return; }
    const int W = p.W, H = p.H, HW = W * H;
    __shared__ float red[PREP_WARPS][3 * LMAX];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int w = (blockIdx.x - 1) * PREP_WARPS + warp;
    const bool active = w < strips * chunks;
    const int cy = w / strips, sx = w - cy * strips;
    const int gx = sx * PREP_COLS + lane;
    const int gxc = gx < W ? gx : W - 1;
    const bool own_col = active && lane < PREP_COLS && gx < W;
    const bool has_right = own_col && gx + 1 < W;
    const int Y0 = active ? cy * PREP_ROWS : 0;
    int yo[PREP_ROWS + 1];                                   // clamped row offsets
#pragma unroll
    for (int r = 0; r <= PREP_ROWS; ++r) yo[r] = min(Y0 + r, H - 1) * W;

    // ---- phase 1: every load of the patch (target rows, the disparity taps of all scales) ----
    float t[PREP_ROWS + 1][C];
    if (do_stats) {
        const float* tg = p.tgt + (long long)n * p.tgt_ns + gxc;
#pragma unroll
        for (int r = 0; r <= PREP_ROWS; ++r)
#pragma unroll
            for (int c = 0; c < C; ++c) t[r][c] = __ldg(tg + c * HW + yo[r]);
    }
    // native scale: q[l][r] = disparity of row r; low-res scale: q[l][2k], q[l][2k+1] = the two horizontal
    // taps of low-res row yb + k (k = 0..3: a 5-row patch touches at most 4 rows at scale <= 1/2)
    float q[LMAX][8], fxu[LMAX];
    int yb[LMAX];
    bool native[LMAX], use[LMAX];
#pragma unroll
    for (int l = 0; l < LMAX; ++l) {
        native[l] = true; use[l] = false; fxu[l] = 0.f; yb[l] = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) q[l][k] = 0.f;
        if (l < p.L) {
            const int dw = p.dw[l], dh = p.dh[l];
            native[l] = (dw == W && dh == H);
            use[l] = !native[l] || do_stats;
            if (native[l]) {
                if (do_stats) {
                    const float* dp = p.disp[l] + (long long)n * HW + gxc;
#pragma unroll
                    for (int r = 0; r <= PREP_ROWS; ++r) q[l][r] = __ldg(dp + yo[r]);
                }
            } else {
                int xa0, xa1, yb1; float fy0;
                up_taps(gxc, dw, W, xa0, xa1, fxu[l]);
                up_taps(min(Y0, H - 1), dh, H, yb[l], yb1, fy0);
                const float* dp = p.disp[l] + (long long)n * dw * dh;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float* rw = dp + min(yb[l] + k, dh - 1) * dw;
                    q[l][2 * k] = __ldg(rw + xa0); q[l][2 * k + 1] = __ldg(rw + xa1);
                }
            }
        }
    }

    // ---- phase 2: edge weights of the patch (shared by the scales): wx[r] between columns gx, gx+1 of
    // row r, wy[r] between rows r-1 and r; the ownership masks are folded into the weights ----
    float wx[PREP_ROWS], wy[PREP_ROWS + 1];
    if (do_stats) {
#pragma unroll
        for (int r = 0; r <= PREP_ROWS; ++r) {
            float gxv = 0.f, gyv = 0.f;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                if (r < PREP_ROWS) gxv += fabsf(t[r][c] - __shfl_down_sync(0xffffffffu, t[r][c], 1));
                if (r > 0) gyv += fabsf(t[r - 1][c] - t[r][c]);
            }
            if (r < PREP_ROWS) wx[r] = (has_right && Y0 + r < H) ? __expf(-gxv * (1.0f / C)) : 0.f;
            wy[r] = (r > 0 && own_col && Y0 + r < H) ? __expf(-gyv * (1.0f / C)) : 0.f;
        }
    }
#pragma unroll
    for (int l = 0; l < LMAX; ++l) {
        if (!use[l]) continue;
        float d[PREP_ROWS + 1];
        if (native[l]) {
#pragma unroll
            for (int r = 0; r <= PREP_ROWS; ++r) d[r] = q[l][r];
        } else {
            const int dh = p.dh[l];
            float h[4];                                      // low-res rows yb .. yb+3, interpolated horizontally
#pragma unroll
            for (int k = 0; k < 4; ++k) h[k] = fmaf(fxu[l], q[l][2 * k + 1] - q[l][2 * k], q[l][2 * k]);
            float* out = const_cast<float*>(p.dfull[l]) + (long long)n * HW + gx;
#pragma unroll
            for (int r = 0; r <= PREP_ROWS; ++r) {
                int ya0, ya1; float fyu;
                up_taps(min(Y0 + r, H - 1), dh, H, ya0, ya1, fyu);
                const float top = sel4(h, ya0 - yb[l]), bot = sel4(h, ya1 - yb[l]);
                d[r] = fmaf(fyu, bot - top, top);
                if (r < PREP_ROWS && Y0 + r < H && own_col) out[yo[r]] = d[r];
            }
        }
        if (do_stats) {
            float v0 = 0.f, v1 = 0.f, v2 = 0.f;
#pragma unroll
            for (int r = 0; r <= PREP_ROWS; ++r) {
                if (r < PREP_ROWS) {
                    const float dr = __shfl_down_sync(0xffffffffu, d[r], 1);
                    v0 = fmaf(fabsf(d[r] - dr), wx[r], v0);
                    v2 += (own_col && Y0 + r < H) ? d[r] : 0.f;
                }
                if (r > 0) v1 = fmaf(fabsf(d[r - 1] - d[r]), wy[r], v1);   // rows r-1 (owned) and r
            }
            v0 = warp_sum(v0); v1 = warp_sum(v1); v2 = warp_sum(v2);
            if (lane == 0) { red[warp][3 * l] = v0; red[warp][3 * l + 1] = v1; red[warp][3 * l + 2] = v2; }
        }
    }
    if (!do_stats) return;
    __syncthreads();
    if ((int)threadIdx.x < 3 * p.L) {
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < PREP_WARPS; ++k) s += red[k][threadIdx.x];
        const int l = threadIdx.x / 3, k = threadIdx.x - 3 * l;
        part[(((long long)l * p.N + n) * nblk + (blockIdx.x - 1)) * 4 + k] = s;
    }
}

// Transpose-reduce of 16 values per lane: afterwards lanes k and k + 16 hold the warp total of value k (17 shuffles)
__device__ __forceinline__ float warp_reduce_16(float (&v)[16]) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int half = 8; half >= 1; half >>= 1) {
        const bool up = (lane & half) != 0;
#pragma unroll
        for (int i = 0; i < half; ++i) {
            const float send = up ? v[i] : v[i + half];
            const float keep = up ? v[i + half] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, half);
        }
    }
    return v[0] + __shfl_xor_sync(0xffffffffu, v[0], 16);
}

// The same patch work for the usual decoder layout, specialised and written lean (the generic kernel above spends most
// of its instructions on per-scale bookkeeping): scales 0 .. NLOW-1 are low-resolution, scale NLOW (the last) is at
// full resolution, the call is the fused fwd+bwd one (statistics wanted), 3 (NLOW + 1) <= 16.
template <int C, int NLOW>
__global__ void __launch_bounds__(32 * PREP_WARPS, MD2_PREP_MINB) prep_fast_kernel(const __grid_constant__ FusedParams p, int strips, int chunks,
                                                                    int nblk, float* __restrict__ pose_ab,
                                                                    float* __restrict__ part, int zero_blocks) {
    constexpr int NS = NLOW + 1;
    static_assert(3 * NS <= 16, "one transpose-reduce of 16 values");
    const int n = blockIdx.y;
    pdl_trigger();
    if (blockIdx.x == 0 || (int)blockIdx.x > nblk) { prep_pose_or_zero<C>(p, nblk, pose_ab, zero_blocks); return; }
    __shared__ float red[PREP_WARPS][16];
    __shared__ float hrow[PREP_WARPS][4][32];               // the four horizontally interpolated low-res rows of a patch, per lane
    const int W = p.W, H = p.H, HW = W * H;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int w = (blockIdx.x - 1) * PREP_WARPS + warp;
    const bool active = w < strips * chunks;
    const int cy = w / strips, sx = w - cy * strips;
    const int gx = sx * PREP_COLS + lane;
    const int gxc = gx < W ? gx : W - 1;
    const bool own_col = active && lane < PREP_COLS && gx < W;
    const bool has_right = own_col && gx + 1 < W;
    const int Y0 = active ? cy * PREP_ROWS : 0;
    int yo[PREP_ROWS + 1];                                   // clamped row offsets
    float rowm[PREP_ROWS + 1];                               // 1 for rows of this patch that are inside the image
#pragma unroll
    for (int r = 0; r <= PREP_ROWS; ++r) { yo[r] = min(Y0 + r, H - 1) * W; rowm[r] = (Y0 + r < H) ? 1.f : 0.f; }

    // ---- every load of the patch ----
    const float* tg = p.tgt + ((long long)n * p.tgt_ns + gxc);
    float t[PREP_ROWS + 1][C], dnat[PREP_ROWS + 1];
#pragma unroll
    for (int r = 0; r <= PREP_ROWS; ++r)
#pragma unroll
        for (int c = 0; c < C; ++c) t[r][c] = __ldg(tg + (c * HW + yo[r]));
    {
        const float* dp = p.disp[NLOW] + ((long long)n * HW + gxc);
#pragma unroll
        for (int r = 0; r <= PREP_ROWS; ++r) dnat[r] = __ldg(dp + yo[r]);
    }
    float q[NLOW > 0 ? NLOW : 1][8], fxu[NLOW > 0 ? NLOW : 1];
    int yb[NLOW > 0 ? NLOW : 1];
#pragma unroll
    for (int l = 0; l < NLOW; ++l) {
        const int dw = p.dw[l], dh = p.dh[l];
        int xa0, xa1, yb1; float fy0;
        tap_load(p.tap_x[l], gxc, xa0, xa1, fxu[l]);
        tap_load(p.tap_y[l], min(Y0, H - 1), yb[l], yb1, fy0);
        const float* dp = p.disp[l] + (long long)n * dw * dh;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int ro = min(yb[l] + k, dh - 1) * dw;
            q[l][2 * k] = __ldg(dp + (ro + xa0)); q[l][2 * k + 1] = __ldg(dp + (ro + xa1));
        }
    }

    // ---- edge weights (shared by the scales), ownership masks folded in ----
    float wx[PREP_ROWS], wy[PREP_ROWS + 1];
    const float mcol = own_col ? 1.f : 0.f, mright = has_right ? 1.f : 0.f;
#pragma unroll
    for (int r = 0; r <= PREP_ROWS; ++r) {
        float gxv = 0.f, gyv = 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            if (r < PREP_ROWS) gxv += fabsf(t[r][c] - __shfl_down_sync(0xffffffffu, t[r][c], 1));
            if (r > 0) gyv += fabsf(t[r - 1][c] - t[r][c]);
        }
        if (r < PREP_ROWS) wx[r] = __expf(-gxv * (1.0f / C)) * (mright * rowm[r]);
        wy[r] = r > 0 ? __expf(-gyv * (1.0f / C)) * (mcol * rowm[r]) : 0.f;
    }

    // ---- per scale: full-resolution disparities of the patch, scratch, sums ----
    float v[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) v[k] = 0.f;
#pragma unroll
    for (int l = 0; l < NS; ++l) {
        float d[PREP_ROWS + 1];
        if (l == NLOW) {
#pragma unroll
            for (int r = 0; r <= PREP_ROWS; ++r) d[r] = dnat[r];
        } else {
            // low-res rows yb .. yb+3, interpolated horizontally, parked in this lane's column of shared memory: the rows a
            // full-resolution row needs are picked by a warp-uniform index (no select chains, no barrier: lane-private)
            __syncwarp();
#pragma unroll
            for (int k = 0; k < 4; ++k) hrow[warp][k][lane] = fmaf(fxu[l], q[l][2 * k + 1] - q[l][2 * k], q[l][2 * k]);
            __syncwarp();
            float* out = const_cast<float*>(p.dfull[l]) + ((long long)n * HW + gx);
#pragma unroll
            for (int r = 0; r <= PREP_ROWS; ++r) {
                int ya0, ya1; float fyu;
                tap_load(p.tap_y[l], min(Y0 + r, H - 1), ya0, ya1, fyu);
                const float top = hrow[warp][(ya0 - yb[l]) & 3][lane], bot = hrow[warp][(ya1 - yb[l]) & 3][lane];
                d[r] = fmaf(fyu, bot - top, top);
                if (r < PREP_ROWS && Y0 + r < H && own_col) out[yo[r]] = d[r];
            }
        }
#pragma unroll
        for (int r = 0; r <= PREP_ROWS; ++r) {
            if (r < PREP_ROWS) {
                const float dr = __shfl_down_sync(0xffffffffu, d[r], 1);
                v[3 * l] = fmaf(fabsf(d[r] - dr), wx[r], v[3 * l]);
                v[3 * l + 2] = fmaf(d[r], mcol * rowm[r], v[3 * l + 2]);
            }
            if (r > 0) v[3 * l + 1] = fmaf(fabsf(d[r - 1] - d[r]), wy[r], v[3 * l + 1]);   // rows r-1 (owned) and r
        }
    }
    const float tot = warp_reduce_16(v);
    if (lane < 16) red[warp][lane] = tot;
    __syncthreads();
    if ((int)threadIdx.x < 3 * NS) {
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < PREP_WARPS; ++k) s += red[k][threadIdx.x];
        const int l = threadIdx.x / 3, k = threadIdx.x - 3 * l;
        part[(((long long)l * p.N + n) * nblk + (blockIdx.x - 1)) * 4 + k] = s;
    }
}

// ------------------------------------------------------------------------------------------
// the marching-warp kernel (md2_march.cuh), persistent: one-warp blocks, as many as are resident
// on the whole GPU; block b walks the work items (strip, chunk, scale, image) b, b + grid, ...  The last warp to finish an item of a (scale, image) reduces that group's
// partial sums in a fixed order, the very last one finalises the loss and the pose gradients
// (deterministic loss).
// ------------------------------------------------------------------------------------------
#ifndef MD2_ROLE_SWAP
#define MD2_ROLE_SWAP 1
#endif
template <int C, int S, bool BWD>
struct MarchCfg {
    // register budget per thread; registers are allocated per warp in units of 512, so the useful
    // tiers are 96 (20 resident warps per SM), 112 (18), 128 (16), 144 (14), 160 (12), 192 (10)
#ifndef MD2_MAXREG_C1   // (overridable for tuning experiments)
#define MD2_MAXREG_C1 128
#endif
#ifndef MD2_MAXREG_C3
#define MD2_MAXREG_C3 192
#endif
    static constexpr int MAXREG = C == 1 ? MD2_MAXREG_C1 : MD2_MAXREG_C3;
};

template <int C, int S, bool BWD>
__global__ void __maxnreg__((MarchCfg<C, S, BWD>::MAXREG))
march_kernel(const __grid_constant__ FusedParams p, int strips, int chunks, int q_full, int lgroups) {
    extern __shared__ __align__(16) float wsm[];
    using M = March<C, S, BWD>;
    constexpr int NP = M::NPART;
    const int lane = threadIdx.x & 31;
    int role = threadIdx.x >> 5;            // 0: warp F (forward), 1: warp B (backward)
    pdl_trigger();
    pdl_wait();
    // segments = (strip, chunk) of a (scale, image); an item is one full-height chunk, or -- when the image
    // height is not a multiple of the chunk height -- a group of short last chunks of neighbouring strips (the
    // `strips` short chunks of a (scale, image) are cut into `lgroups` groups), so that all items are about
    // equally long and their number matches the resident blocks of the GPU
    const int ipg = strips * chunks;                     // segments (= partial-sum rows) per (scale, image)
    const int n_full = strips * q_full;
    const int ipi = n_full + (chunks > q_full ? lgroups : 0);   // items per (scale, image)
    const int LN = p.L * p.N;
    const int items = ipi * LN;
    int gslot = 0;
    if (BWD) {
        // The two warps of a block sit on neighbouring schedulers (warp slots 2k, 2k+1 of the SM).  With a fixed role per
        // warp index every warp F (the heavier role) would land on an even scheduler: swap the roles in every other pair
        // of blocks on an SM (bit 2 of the hardware warp slot), so that each scheduler gets as many F as B warps.
        int* swap_flag = reinterpret_cast<int*>(wsm + M::SMEM_FLOATS - 2);
        if (threadIdx.x == 0) {
#pragma unroll
            for (int b = 0; b < MARCH_NBAR; ++b) mb_init(bar_ref_of(wsm + M::RING_FLOATS), b, 32);
            unsigned int wid;
            asm volatile("mov.u32 %0, %%warpid;" : "=r"(wid));
            *swap_flag = MD2_ROLE_SWAP ? (int)((wid >> 2) & 1u) : 0;
        }
        __syncthreads();
        role ^= *swap_flag;
    }
    // one warp pair per block, item index from blockIdx only, so that everything derived from it is
    // warp-uniform for the compiler (uniform registers / constant-bank operands); the grid is
    // at most the number of blocks resident on the whole GPU
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
        const int z = it / ipi, rem = it - z * ipi;
        int cy, sx, sx_end;
        if (rem < n_full) { cy = rem / strips; sx = rem - cy * strips; sx_end = sx + 1; }
        else { cy = q_full; sx = (rem - n_full) * strips / lgroups; sx_end = (rem - n_full + 1) * strips / lgroups; }
        for (; sx < sx_end; ++sx) {
            float v[32];
            if (role == 0) M::run_forward(p, sx, cy, z, lane, wsm, gslot, v);
            else M::run_backward(p, sx, cy, z, lane, wsm, gslot, v);
            const float tot = warp_reduce_32(v);
            // warp F owns the loss sums [0, NSTAT), warp B the pose sums [NSTAT, NP)
            if (role == 0 ? lane < (BWD ? NSTAT : NP) : (lane >= NSTAT && lane < NP))
                p.partial[((long long)z * ipg + cy * strips + sx) * NP + lane] = tot;
            if (BWD) __syncthreads();   // both warps are done with the ring before the next segment reuses it
        }
    }
}

// ------------------------------------------------------------------------------------------
// the single-warp marching kernel (md2_march2.cuh): value + gradient.  Persistent one-warp blocks, as many as are
// resident on the whole GPU; block b walks the work items b, b + grid, ... (same items / partial-sum rows as above)
// ------------------------------------------------------------------------------------------
template <int C, int S, bool AM, bool DBG, bool GRAD>
__global__ void __maxnreg__((March2<C, S, AM, DBG, GRAD>::MAXREG))
march2_kernel(const __grid_constant__ FusedParams p, int strips, int chunks, int q_full, int lgroups) {
    extern __shared__ __align__(16) float wsm[];
    using M = March2<C, S, AM, DBG, GRAD>;
    constexpr int NP = M::NPART;
    const int lane = threadIdx.x;
    pdl_trigger();
    pdl_wait();                                          // the prep kernel's outputs (poses, upsampled disparities, sums)
    const int ipg = strips * chunks;                     // segments (= partial-sum rows) per (scale, image)
    const int n_full = strips * q_full;
    const int ipi = n_full + (chunks > q_full ? lgroups : 0);   // items per (scale, image)
    const int items = ipi * p.L * p.N;
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
        const int z = it / ipi, rem = it - z * ipi;
        int cy, sx, sx_end;
        if (rem < n_full) { cy = rem / strips; sx = rem - cy * strips; sx_end = sx + 1; }
        else { cy = q_full; sx = (rem - n_full) * strips / lgroups; sx_end = (rem - n_full + 1) * strips / lgroups; }
        for (; sx < sx_end; ++sx) {
            float v[32];
            M::run(p, sx, cy, z, lane, wsm, v);
            const float tot = warp_reduce_32(v);
            // value + gradient: the loss sum and the pose sums (the smoothness sums come from the prep kernel); forward-only: the four statistics
            if (GRAD ? (lane == 0 || (lane >= NSTAT && lane < NP)) : lane < NSTAT)
                p.partial[((long long)z * ipg + cy * strips + sx) * NP + lane] = tot;
        }
    }
}

// ------------------------------------------------------------------------------------------
// finish kernel (one launch after the marching kernel); every block is independent, all sums
// are taken in a fixed order (deterministic), nothing is atomic:
//   block 0             per-(scale, image) loss sums from the per-item partials (and, for the fused
//                       fwd+bwd call, the smoothness sums from the prep kernel's partials) ->
//                       statistics, saved statistics, loss scalar
//   blocks 1 .. S*N     (backward) pose gradient of one (source, image): G | h summed over all
//                       scales and items in double, then the K / composeT / so3 adjoints
//   remaining blocks    (backward, low-res decoder scales) adjoint of the upsample, gather form,
//                       separable: one block per low-res output row (low_rows = sum of the low-res
//                       heights, per image).  Phase A sums the contributing full-resolution rows
//                       with their vertical weights into shared memory (128-bit coalesced loads),
//                       phase B the contributing columns per low-res pixel.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// called once by every (source, image) after it wrote its row of k.part: true for the last of the S*N arrivals, which then
// forms grad_K / grad_invK and resets the counter (so a replayed graph finds it at 0 again)
__device__ __forceinline__ bool intrinsics_last(const IntrIO& k, int S, int N) {
    __threadfence();
    const bool last = atomicAdd(k.count, 1u) == (unsigned)(S * N - 1);
    if (last) __threadfence();
    return last;
}

constexpr int FIN_MAXROWS = 64;   // contributing full-resolution rows handled per pass of phase A
constexpr int FIN_THREADS = 128;
#ifndef MD2_FIN_MINB
#define MD2_FIN_MINB 7
#endif
#ifndef MD2_FIN_UNROLL
#define MD2_FIN_UNROLL 16
#endif
constexpr int FIN_UNROLL = MD2_FIN_UNROLL;
#ifndef MD2_FIN_TIMING   // timing experiments only (wrong results): 1 = no pose finalisation, 2 = no pose blocks, 3 = no adjoint blocks, 4 = no loss block
#define MD2_FIN_TIMING 0
#endif  // small blocks: the whole grid is resident at once (one latency chain, no waves)

__global__ void __launch_bounds__(FIN_THREADS, MD2_FIN_MINB) finish_kernel(const __grid_constant__ FusedParams p, int NP, int ipg, int bwd, int low_rows,
                                                                           const __grid_constant__ IntrIO intr) {
    extern __shared__ __align__(16) float vrow[];   // [W rounded up to 4] (adjoint blocks)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    pdl_wait();
    const int LN = p.L * p.N;
    int b = blockIdx.x;
    if (b == 0) {
        if (p.mode == 1 || MD2_FIN_TIMING == 4) return;
        // FIN_THREADS / 32 ... lanes per (scale, image) group: strided partial sums with the loads issued in unrolled batches
        // (a rolled loop would pay one L2 round trip per iteration), then a fixed-order butterfly over the lanes of a group
        constexpr int GL = 4;                                 // lanes per group
        const int sub = threadIdx.x & (GL - 1);
        for (int z0 = 0; z0 < LN; z0 += FIN_THREADS / GL) {
            const int z = z0 + (threadIdx.x / GL);
            float v[4] = {0.f, 0.f, 0.f, 0.f};
            if (z < LN) {
                const float* pp = p.partial + (long long)z * ipg * NP;
                if (p.mode == 0) {                            // forward-only: warp F also carries the smoothness sums
#pragma unroll 4
                    for (int it = sub; it < ipg; it += GL) {
#pragma unroll
                        for (int k = 0; k < 4; ++k) v[k] += __ldcg(pp + (long long)it * NP + k);
                    }
                } else {
#pragma unroll 8
                    for (int it = sub; it < ipg; it += GL) v[0] += __ldcg(pp + (long long)it * NP);
                    const float4* q = reinterpret_cast<const float4*>(p.prep_part) + (long long)z * p.prep_nblk;
#pragma unroll 8
                    for (int it = sub; it < p.prep_nblk; it += GL) {
                        const float4 t = __ldcg(q + it);
                        v[1] += t.x; v[2] += t.y; v[3] += t.z;
                    }
                }
            }
#pragma unroll
            for (int o = GL / 2; o > 0; o >>= 1)
#pragma unroll
                for (int k = 0; k < 4; ++k) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
            if (z < LN && sub == 0) {
                float* st = p.stats_out + (long long)z * NSTAT;
#pragma unroll
                for (int k = 0; k < NSTAT; ++k) st[k] = v[k];
                if (p.saved && p.saved != p.stats_out)
#pragma unroll
                    for (int k = 0; k < NSTAT; ++k) p.saved[(long long)z * NSTAT + k] = v[k];
            }
        }
        __syncthreads();
        // loss = loss_scale * sum_i [ mean(warp_loss_i) + smooth_w_i * smooth_loss(dhat_i, target) ]
        // (src/training.jl:64-69,77; same terms as loss_from_stats): one lane per (scale, image), double
        if (warp == 0 && p.loss) {
            const double P = (double)p.W * p.H;
            const double cx = 1.0 / ((double)(p.W - 1) * p.H * p.N), cy = 1.0 / ((double)p.W * (p.H - 1) * p.N);
            const double rPN = 1.0 / (P * p.N);
            double acc = 0.0;
            for (int z = lane; z < LN; z += 32) {
                const float* st = p.stats_out + (long long)z * NSTAT;
                const double m = p.normalize_disp ? ((double)st[3] / P + 1e-7) : 1.0;
                acc += (double)st[0] * rPN + (double)p.smooth_w[z / p.N] * (cx * st[1] + cy * st[2]) / m;
            }
            acc = warp_sum_d(acc);
            if (lane == 0) *p.loss = (float)(acc * p.loss_scale);
        }
        return;
    }
    b -= 1;
    if (!bwd) return;
    if (b < p.S * p.N) {
        if (MD2_FIN_TIMING == 2) return;
        // pose gradient of (source s, image nn): 12 sums over all scales and segments.  Three lanes per row (one float4
        // each; NP and NSTAT are multiples of 4), FIN_PR row groups, loads issued in unrolled batches; then 12 threads add
        // the row-group partials in order, in double
        constexpr int FIN_PR = FIN_THREADS / 3;
        __shared__ double pacc[FIN_PR][12];
        const int s = b / p.N, nn = b % p.N;
        const int q4 = threadIdx.x % 3, j = threadIdx.x / 3;
        if (j < FIN_PR) {
            double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
            const int rows = p.L * ipg;
#pragma unroll 4
            for (int r = j; r < rows; r += FIN_PR) {
                const int l = r / ipg, it = r - l * ipg;
                const float4 t = __ldcg(reinterpret_cast<const float4*>(p.partial + (((long long)l * p.N + nn) * ipg + it) * NP + NSTAT + 12 * s) + q4);
                a0 += (double)t.x; a1 += (double)t.y; a2 += (double)t.z; a3 += (double)t.w;
            }
            pacc[j][4 * q4] = a0; pacc[j][4 * q4 + 1] = a1; pacc[j][4 * q4 + 2] = a2; pacc[j][4 * q4 + 3] = a3;
        }
        __syncthreads();
        if (threadIdx.x < 12) {
            double a = 0.0;
#pragma unroll 6
            for (int q = 0; q < FIN_PR; ++q) a += pacc[q][threadIdx.x];
            pacc[0][threadIdx.x] = a;
        }
        __syncthreads();
        __shared__ int last;
        if (threadIdx.x == 0) {
            last = 0;
            if (MD2_FIN_TIMING != 1) {
                finalize_pose(p.pose, s, nn, &pacc[0][0], &pacc[0][0] + 9);
                if (intr.part) {   // (a separate kernel parameter: FusedParams, which the marching kernels read, keeps its layout)
                    intrinsics_part(p.pose, s, nn, &pacc[0][0], &pacc[0][0] + 9, intr.part + 18 * (long long)b);
                    last = intrinsics_last(intr, p.S, p.N);
                }
            }
        }
        if (intr.part) {   // (uniform: a launch parameter) the last pose block sums the intrinsics gradients, one element per thread
            __syncthreads();
            if (!last) return;
            const int ne = 18 * (p.pose.kstride ? p.N : 1);
            for (int e = threadIdx.x; e < ne; e += blockDim.x) reduce_intrinsics_elem(intr, p.pose.kstride, p.S, p.N, e);
            __syncthreads();
            if (threadIdx.x == 0) *intr.count = 0u;
        }
        return;
    }
    b -= p.S * p.N;
    if (MD2_FIN_TIMING == 3) return;
    // (image, low-res scale, low-res row) of this block: block-uniform scalar code
    const int n = b / low_rows;
    int yi = b - n * low_rows, l = -1;
    for (int k = 0; k < p.L; ++k) {
        if (p.dw[k] == p.W && p.dh[k] == p.H) continue;
        if (yi < p.dh[k]) { l = k; break; }
        yi -= p.dh[k];
    }
    if (l < 0 || n >= p.N) return;
    const int w = p.dw[l], h = p.dh[l];
    const int W = p.W, H = p.H;
    const float* g = p.gfull[l] + (long long)n * W * H;
    __shared__ float wys[FIN_MAXROWS];
    const float* __restrict__ wts = p.inv_w[l];
    // the full-resolution rows that reach low-res row yi and their weights (adjoint tap table: no search, no divisions)
    int ylo, ny, ystart;
    {
        const float4 e = __ldg(reinterpret_cast<const float4*>(p.inv_y[l]) + yi);
        ylo = __float_as_int(e.x); ny = __float_as_int(e.y); ystart = __float_as_int(e.z);
    }
    const bool vec = (W & 3) == 0 && (reinterpret_cast<uintptr_t>(g) & 15) == 0;
    for (int base = 0; base < ny; base += FIN_MAXROWS) {
        __syncthreads();
        if ((int)threadIdx.x < FIN_MAXROWS && base + (int)threadIdx.x < ny) wys[threadIdx.x] = __ldg(wts + ystart + base + threadIdx.x);
        __syncthreads();
        const int cnt = min(FIN_MAXROWS, ny - base);
        if (vec) {
            for (int x = 4 * threadIdx.x; x < W; x += 4 * FIN_THREADS) {
                float4 acc = base ? *reinterpret_cast<const float4*>(vrow + x) : make_float4(0.f, 0.f, 0.f, 0.f);
                const float* gp = g + (long long)(ylo + base) * W + x;
#pragma unroll FIN_UNROLL
                for (int k = 0; k < cnt; ++k) {
                    const float4 q = __ldcg(reinterpret_cast<const float4*>(gp + (long long)k * W));
                    const float wk = wys[k];
                    acc.x = fmaf(wk, q.x, acc.x); acc.y = fmaf(wk, q.y, acc.y);
                    acc.z = fmaf(wk, q.z, acc.z); acc.w = fmaf(wk, q.w, acc.w);
                }
                *reinterpret_cast<float4*>(vrow + x) = acc;
            }
        } else {
            for (int x = threadIdx.x; x < W; x += FIN_THREADS) {
                float acc = base ? vrow[x] : 0.f;
                const float* gp = g + (long long)(ylo + base) * W + x;
#pragma unroll 8
                for (int k = 0; k < cnt; ++k) acc = fmaf(wys[k], __ldcg(gp + (long long)k * W), acc);
                vrow[x] = acc;
            }
        }
    }
    __syncthreads();
    for (int xi = threadIdx.x; xi < w; xi += FIN_THREADS) {
        const float4 e = __ldg(reinterpret_cast<const float4*>(p.inv_x[l]) + xi);
        const int xlo = __float_as_int(e.x), nx = __float_as_int(e.y);
        const float* __restrict__ wx = wts + __float_as_int(e.z);
        float acc = 0.f;
#pragma unroll 4
        for (int k = 0; k < nx; ++k) acc = fmaf(__ldg(wx + k), vrow[xlo + k], acc);
        p.gdisp[l][((long long)n * h + yi) * w + xi] = acc;
    }
}

// ------------------------------------------------------------------------------------------
// host orchestration
// ------------------------------------------------------------------------------------------
// blocks (warp F [+ warp B]) of march_kernel<C,S,BWD> resident per SM (occupancy API, cached)
template <int C, int S, bool BWD>
static int march_resident() {
    using M = March<C, S, BWD>;
    static int resident = 0;
    if (!resident) {
        const size_t smem = sizeof(float) * (size_t)M::SMEM_FLOATS;
        int occ = 0;
        if (cudaFuncSetAttribute(march_kernel<C, S, BWD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) occ = 0;
        cudaFuncSetAttribute(march_kernel<C, S, BWD>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, march_kernel<C, S, BWD>, M::THREADS, smem) != cudaSuccess) occ = 0;
        resident = occ > 0 ? occ : 8;
        if (getenv("MD2_DEBUG")) fprintf(stderr, "[md2] march_kernel<%d,%d,%d>: %d resident blocks/SM, %zu B smem/block\n", C, S, (int)BWD, resident, smem);
    }
    return resident;
}

template <int C, int S, bool BWD>
static int launch_march(md2_ctx* ctx, const FusedParams& p, cudaStream_t st) {
    using M = March<C, S, BWD>;
    const size_t smem = sizeof(float) * (size_t)M::SMEM_FLOATS;
    const int strips = cdiv(p.W, M::OW), chunks = cdiv(p.H, p.m_R), q_full = p.H / p.m_R;
    const int lgroups = p.m_group > 0 ? (p.m_group < strips ? p.m_group : strips) : 1;
    const long long items = ((long long)strips * q_full + (chunks > q_full ? lgroups : 0)) * p.L * p.N;
    const long long cap = (long long)ctx->sm_count * march_resident<C, S, BWD>();
    const int blocks = (int)(items < cap ? items : cap);
    MD2_CHECK(launch_after(1, march_kernel<C, S, BWD>, dim3(blocks), dim3(M::THREADS), smem, st, p, strips, chunks, q_full, lgroups));
    MD2_LAUNCH_CHECK(ctx);
    return 0;
}

template <int C, int S, bool AM, bool DBG = false, bool GRAD = true>
static int march2_resident() {
    using M = March2<C, S, AM, DBG, GRAD>;
    static int resident = 0;
    if (!resident) {
        const size_t smem = sizeof(float) * (size_t)M::SMEM_FLOATS;
        int occ = 0;
        if (cudaFuncSetAttribute(march2_kernel<C, S, AM, DBG, GRAD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) occ = 0;
        // value + gradient: 16 rings of 12 KB need the whole shared-memory carve-out; forward-only: 2 KB per warp -- leave the rest
        // of the 256 KB to the L1 (the gathers of the sources live there)
        cudaFuncSetAttribute(march2_kernel<C, S, AM, DBG, GRAD>, cudaFuncAttributePreferredSharedMemoryCarveout,
                             GRAD ? (int)cudaSharedmemCarveoutMaxShared : 30);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, march2_kernel<C, S, AM, DBG, GRAD>, M::THREADS, smem) != cudaSuccess) occ = 0;
        resident = occ > 0 ? occ : 8;
        if (getenv("MD2_DEBUG")) fprintf(stderr, "[md2] march2_kernel<%d,%d>: %d resident warps/SM, %zu B smem/warp\n", C, S, resident, smem);
    }
    return resident;
}

template <int C, int S, bool AM, bool DBG = false, bool GRAD = true>
static int launch_march2(md2_ctx* ctx, const FusedParams& p, cudaStream_t st) {
    using M = March2<C, S, AM, DBG, GRAD>;
    const size_t smem = sizeof(float) * (size_t)M::SMEM_FLOATS;
    const int strips = cdiv(p.W, M::OW), chunks = cdiv(p.H, p.m_R), q_full = p.H / p.m_R;
    const int lgroups = p.m_group > 0 ? (p.m_group < strips ? p.m_group : strips) : 1;
    const long long items = ((long long)strips * q_full + (chunks > q_full ? lgroups : 0)) * p.L * p.N;
    const long long cap = (long long)ctx->sm_count * march2_resident<C, S, AM, DBG, GRAD>();
    const int blocks = (int)(items < cap ? items : cap);
    MD2_CHECK(launch_after(1, march2_kernel<C, S, AM, DBG, GRAD>, dim3(blocks), dim3(M::THREADS), smem, st, p, strips, chunks, q_full, lgroups));
    MD2_LAUNCH_CHECK(ctx);
    return 0;
}

static int dispatch_march2(md2_ctx* ctx, int C, int S, const FusedParams& p, cudaStream_t st, bool grad = true) {
    const bool am = p.automask != nullptr;
    if (!grad) {   // forward-only instantiations
        if (C == 1 && S == 1) return am ? launch_march2<1, 1, true, false, false>(ctx, p, st) : launch_march2<1, 1, false, false, false>(ctx, p, st);
        if (C == 1 && S == 2) return am ? launch_march2<1, 2, true, false, false>(ctx, p, st) : launch_march2<1, 2, false, false, false>(ctx, p, st);
        if (C == 3 && S == 1) return am ? launch_march2<3, 1, true, false, false>(ctx, p, st) : launch_march2<3, 1, false, false, false>(ctx, p, st);
        if (C == 3 && S == 2) return am ? launch_march2<3, 2, true, false, false>(ctx, p, st) : launch_march2<3, 2, false, false, false>(ctx, p, st);
        return set_error("view_synthesis_loss: unsupported C=%d S=%d (C in {1,3}, S in {1,2})", C, S);
    }
    if (p.dbg) {   // test hook (md2.h: debug_choices): the instantiations that also export the decisions
        if (S != 2) return set_error("view_synthesis_loss: debug_choices needs S = 2");
        if (C == 1) return am ? launch_march2<1, 2, true, true>(ctx, p, st) : launch_march2<1, 2, false, true>(ctx, p, st);
        if (C == 3) return am ? launch_march2<3, 2, true, true>(ctx, p, st) : launch_march2<3, 2, false, true>(ctx, p, st);
    }
    if (C == 1 && S == 1) return am ? launch_march2<1, 1, true>(ctx, p, st) : launch_march2<1, 1, false>(ctx, p, st);
    if (C == 1 && S == 2) return am ? launch_march2<1, 2, true>(ctx, p, st) : launch_march2<1, 2, false>(ctx, p, st);
    if (C == 3 && S == 1) return am ? launch_march2<3, 1, true>(ctx, p, st) : launch_march2<3, 1, false>(ctx, p, st);
    if (C == 3 && S == 2) return am ? launch_march2<3, 2, true>(ctx, p, st) : launch_march2<3, 2, false>(ctx, p, st);
    return set_error("view_synthesis_loss: unsupported C=%d S=%d (C in {1,3}, S in {1,2})", C, S);
}

static int march2_resident_of(int C, int S, bool am, bool grad = true) {
    if (!grad) {
        if (am) {
            if (C == 1) return S == 1 ? march2_resident<1, 1, true, false, false>() : march2_resident<1, 2, true, false, false>();
            return S == 1 ? march2_resident<3, 1, true, false, false>() : march2_resident<3, 2, true, false, false>();
        }
        if (C == 1) return S == 1 ? march2_resident<1, 1, false, false, false>() : march2_resident<1, 2, false, false, false>();
        return S == 1 ? march2_resident<3, 1, false, false, false>() : march2_resident<3, 2, false, false, false>();
    }
    if (am) {
        if (C == 1) return S == 1 ? march2_resident<1, 1, true>() : march2_resident<1, 2, true>();
        return S == 1 ? march2_resident<3, 1, true>() : march2_resident<3, 2, true>();
    }
    if (C == 1) return S == 1 ? march2_resident<1, 1, false>() : march2_resident<1, 2, false>();
    return S == 1 ? march2_resident<3, 1, false>() : march2_resident<3, 2, false>();
}

// which kernel runs the value + gradient calls: the single-warp kernel (default) or the two-warp producer / consumer pair
static bool use_march_v1() {
    static const bool v1 = [] { const char* e = getenv("MD2_MARCH_V1"); return e && atoi(e) != 0; }();
    return v1;
}

static int march_resident_of(int C, int S, bool bwd) {
    if (bwd) {
        if (C == 1) return S == 1 ? march_resident<1, 1, true>() : march_resident<1, 2, true>();
        return S == 1 ? march_resident<3, 1, true>() : march_resident<3, 2, true>();
    }
    if (C == 1) return S == 1 ? march_resident<1, 1, false>() : march_resident<1, 2, false>();
    return S == 1 ? march_resident<3, 1, false>() : march_resident<3, 2, false>();
}

template <bool BWD>
static int dispatch_march(md2_ctx* ctx, int C, int S, const FusedParams& p, cudaStream_t st) {
    if (C == 1 && S == 1) return launch_march<1, 1, BWD>(ctx, p, st);
    if (C == 1 && S == 2) return launch_march<1, 2, BWD>(ctx, p, st);
    if (C == 3 && S == 1) return launch_march<3, 1, BWD>(ctx, p, st);
    if (C == 3 && S == 2) return launch_march<3, 2, BWD>(ctx, p, st);
    return set_error("view_synthesis_loss: unsupported C=%d S=%d (C in {1,3}, S in {1,2})", C, S);
}

// rows per chunk of the marching kernel.  Long chunks amortise the 2*HALO warm-up rows; the item
// count should fill the resident warps of all SMs evenly (one block per SM, `warps` warps each):
// time ~ max(throughput term, longest per-warp chain), both in row-iterations.
static int choose_march_rows_uncached(int W, int H, int LN, bool bwd, int sms, int warps, int& group);
static int choose_march_rows(int W, int H, int LN, bool bwd, int sms, int warps, int& group) {
    // (the search below is a few hundred divisions: remembered per shape, the calls of a training loop repeat it)
    struct Memo { int W, H, LN, bwd, sms, warps, R, group; };
    static thread_local Memo memo[8];
    static thread_local int used = 0, next = 0;
    for (int i = 0; i < used; ++i) {
        const Memo& m = memo[i];
        if (m.W == W && m.H == H && m.LN == LN && m.bwd == (int)bwd && m.sms == sms && m.warps == warps) { group = m.group; return m.R; }
    }
    const int R = choose_march_rows_uncached(W, H, LN, bwd, sms, warps, group);
    memo[next] = Memo{W, H, LN, (int)bwd, sms, warps, R, group};
    next = (next + 1) % 8;
    if (used < 8) ++used;
    return R;
}
static int choose_march_rows_uncached(int W, int H, int LN, bool bwd, int sms, int warps, int& group) {
    static const int env = [] { const char* e = getenv("MD2_MARCH_ROWS"); return e ? atoi(e) : 0; }();
    static const int env_group = [] { const char* e = getenv("MD2_MARCH_GROUP"); return e ? atoi(e) : -1; }();
    const int ow = bwd ? 28 : 30, halo = bwd ? 2 : 1;
    const int strips = cdiv(W, ow);
    const long long base = (long long)strips * LN;
    const double over = 2 * halo + 1.5;                      // warm-up rows + set-up of a segment, in row-iterations
    int best_R = H;
    double best = 1e30;
    group = 1;
    for (int R = H; R >= 8 || R == H; --R) {
        if (env > 0 && R != (env < H ? env : H)) continue;
        const int q = H / R, rem = H % R;
        // short last chunks are grouped so that a group is about as long as a full chunk (measured: cutting them
        // into more, shorter groups to fill every resident block slot is slower: 81.5 vs 77.7 us at 416x128x8)
        int lg = 1;
        if (rem) {
            if (rem < 8 && env <= 0) continue;
            int k = (int)((R + over) / (rem + over));
            if (k < 1) k = 1;
            if (k > strips) k = strips;
            lg = cdiv(strips, k);
            if (env_group >= 1) lg = env_group < strips ? env_group : strips;
        }
        const long long items = base * q + (rem ? (long long)LN * lg : 0);
        const double longest = rem ? fmax(R + over, cdiv(strips, lg) * (rem + over)) : R + over;
        const double total = (double)base * q * (R + over) + (rem ? (double)base * (rem + over) : 0.0);
        const long long per_sm = (items + sms - 1) / sms;
        const double thr = total / ((double)sms * warps);
        const double chain = (double)((per_sm + warps - 1) / warps) * longest;
        const double cost = thr > chain ? thr : chain;
        if (cost < best - 1e-9) { best = cost; best_R = R; group = lg; }
        if (R == 8) break;
    }
    return best_R;
}

// Tap tables of the align-corners upsample (A17) for the low-resolution scales of a shape: computed on the host with the
// very function the kernels used to call per pixel (up_taps: exact integer arithmetic, one division per call), uploaded
// once and kept per shape.  Read-only afterwards, so all streams / workspace banks share them.
struct TapsEntry {
    int W, H, L, dw[MAX_L], dh[MAX_L];
    int wcount[MAX_L] = {};   // floats of the inverse weight list of every low-res scale
    float* dev = nullptr;
    uint64_t last_use = 0;
};
struct TapsCache {
    static constexpr int CAP = 8;
    TapsEntry e[CAP];
    int used = 0;
    uint64_t tick = 0;
};
void taps_destroy(md2_ctx* ctx) {
    TapsCache* tc = static_cast<TapsCache*>(ctx->taps);
    if (!tc) return;
    for (int i = 0; i < tc->used; ++i)
        if (tc->e[i].dev) cudaFree(tc->e[i].dev);
    delete tc;
    ctx->taps = nullptr;
}
// fills p.tap_x / p.tap_y; returns non-zero on error
static int taps_get(md2_ctx* ctx, const md2_vsl_desc* d, FusedParams& p, cudaStream_t st) {
    if (!ctx->taps) ctx->taps = new TapsCache();
    TapsCache* tc = static_cast<TapsCache*>(ctx->taps);
    ++tc->tick;
    TapsEntry* hit = nullptr;
    for (int i = 0; i < tc->used && !hit; ++i) {
        TapsEntry& e = tc->e[i];
        if (e.W == d->W && e.H == d->H && e.L == d->L && memcmp(e.dw, d->disp_w, sizeof(int) * d->L) == 0 && memcmp(e.dh, d->disp_h, sizeof(int) * d->L) == 0) hit = &e;
    }
    const int W = d->W, H = d->H;
    if (!hit) {
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone)
            return set_error("internal: tap tables of a new shape requested under stream capture");
        if (tc->used < TapsCache::CAP) hit = &tc->e[tc->used++];
        else {
            hit = &tc->e[0];
            for (int i = 1; i < tc->used; ++i) if (tc->e[i].last_use < hit->last_use) hit = &tc->e[i];
            MD2_CHECK(cudaDeviceSynchronize());              // a launch in flight may still read the evicted table
            cudaFree(hit->dev); hit->dev = nullptr;
            for (int b = 0; b < MD2_WS_BANKS; ++b) ctx->ws_gen[b]++;   // captured graphs hold its address
        }
        // layout per low-res scale: tap_x (4W) | tap_y (4H) | inv_x (4w) | inv_y (4h) | inv_w (weights of x, then of y)
        std::vector<float> h;
        for (int l = 0; l < d->L; ++l) {
            if (d->disp_w[l] == W && d->disp_h[l] == H) continue;
            std::vector<int> i0s[2], i1s[2];
            std::vector<float> fs[2];
            for (int pass = 0; pass < 2; ++pass) {
                const int n = pass ? H : W, m = pass ? d->disp_h[l] : d->disp_w[l];
                i0s[pass].resize(n); i1s[pass].resize(n); fs[pass].resize(n);
                for (int x = 0; x < n; ++x) {
                    up_taps(x, m, n, i0s[pass][x], i1s[pass][x], fs[pass][x]);
                    float e[4] = {0.f, 0.f, fs[pass][x], 0.f};
                    memcpy(&e[0], &i0s[pass][x], 4); memcpy(&e[1], &i1s[pass][x], 4);
                    h.insert(h.end(), e, e + 4);
                }
            }
            std::vector<float> wts;
            for (int pass = 0; pass < 2; ++pass) {
                const int n = pass ? H : W, m = pass ? d->disp_h[l] : d->disp_w[l];
                for (int i = 0; i < m; ++i) {
                    auto wgt = [&](int x) { return (i0s[pass][x] == i ? 1.f - fs[pass][x] : 0.f) + (i1s[pass][x] == i ? fs[pass][x] : 0.f); };
                    int lo = 0, hi = n - 1;
                    while (lo < hi && wgt(lo) == 0.f) ++lo;
                    while (hi > lo && wgt(hi) == 0.f) --hi;
                    const int cnt = hi - lo + 1, start = (int)wts.size();
                    for (int x = lo; x <= hi; ++x) wts.push_back(wgt(x));
                    float e[4] = {0.f, 0.f, 0.f, 0.f};
                    memcpy(&e[0], &lo, 4); memcpy(&e[1], &cnt, 4); memcpy(&e[2], &start, 4);
                    h.insert(h.end(), e, e + 4);
                }
            }
            while (wts.size() & 3) wts.push_back(0.f);       // keep the next scale's tables 16-byte aligned
            h.insert(h.end(), wts.begin(), wts.end());
            hit->wcount[l] = (int)wts.size();
        }
        MD2_CHECK(cudaMalloc(&hit->dev, sizeof(float) * (h.size() + 4)));
        MD2_CHECK(cudaMemcpy(hit->dev, h.data(), sizeof(float) * h.size(), cudaMemcpyHostToDevice));
        hit->W = W; hit->H = H; hit->L = d->L;
        memset(hit->dw, 0, sizeof(hit->dw)); memset(hit->dh, 0, sizeof(hit->dh));
        memcpy(hit->dw, d->disp_w, sizeof(int) * d->L); memcpy(hit->dh, d->disp_h, sizeof(int) * d->L);
    }
    hit->last_use = tc->tick;
    const float* q = hit->dev;
    for (int l = 0; l < d->L; ++l) {
        if (d->disp_w[l] == W && d->disp_h[l] == H) { p.tap_x[l] = p.tap_y[l] = p.inv_x[l] = p.inv_y[l] = p.inv_w[l] = nullptr; continue; }
        p.tap_x[l] = q; q += (size_t)4 * W;
        p.tap_y[l] = q; q += (size_t)4 * H;
        p.inv_x[l] = q; q += (size_t)4 * d->disp_w[l];
        p.inv_y[l] = q; q += (size_t)4 * d->disp_h[l];
        p.inv_w[l] = q; q += (size_t)hit->wcount[l];
    }
    return 0;
}

static int check_desc(const md2_vsl_desc* d, bool need_loss_inputs) {
    MD2_REQUIRE(d != nullptr, "null descriptor");
    MD2_REQUIRE(d->W >= 2 && d->H >= 2 && d->W <= 65535 && d->H <= 32767, "W, H must be in 2..65535 / 2..32767");
    MD2_REQUIRE((long long)d->W * d->H * d->C < (1LL << 31), "one image must have fewer than 2^31 elements");
    MD2_REQUIRE(d->W <= 12288, "W must be <= 12288 (one image row is staged in shared memory)");
    MD2_REQUIRE(d->N >= 1, "N must be >= 1");
    MD2_REQUIRE(d->C == 1 || d->C == 3, "C must be 1 or 3");
    MD2_REQUIRE(d->S >= 1 && d->S <= MAX_S, "S must be 1 or 2");
    MD2_REQUIRE(d->K && d->invK, "K / invK are null (grad_K / grad_invK need them too)");
    MD2_REQUIRE(d->per_image_K == 0 || d->per_image_K == 1, "per_image_K must be 0 (one (3,3) K / invK) or 1 ((3,3,N))");
    for (int s = 0; s < d->S; ++s) {
        MD2_REQUIRE(d->source[s] != nullptr, "null source image");
        MD2_REQUIRE(d->rot[s] && d->trans[s], "null pose");
    }
    if (need_loss_inputs) {
        MD2_REQUIRE(d->L >= 1 && d->L <= MAX_L, "L must be in 1..8");
        MD2_REQUIRE((long long)d->L * d->N <= 65535, "L*N too large");
        MD2_REQUIRE(d->target != nullptr, "null target image");
        for (int l = 0; l < d->L; ++l) {
            MD2_REQUIRE(d->disparity[l] != nullptr, "null disparity");
            const bool native = d->disp_w[l] == d->W && d->disp_h[l] == d->H;
            MD2_REQUIRE(native || (d->disp_w[l] >= 2 && d->disp_h[l] >= 2 && 2 * d->disp_w[l] <= d->W + 1 &&
                                   2 * d->disp_h[l] <= d->H + 1),
                        "a disparity must be full-resolution or at most half-resolution (decoder scales 1/2, 1/4, ...)");
        }
    }
    return 0;
}

static void fill_pose_io(const md2_vsl_desc* d, PoseIO& io) {
    io.mode = d->pose_mode;
    io.K = d->K; io.invK = d->invK;
    io.kstride = d->per_image_K ? 9 : 0;
    for (int s = 0; s < MAX_S; ++s) {
        io.rot[s] = s < d->S ? d->rot[s] : nullptr;
        io.trans[s] = s < d->S ? d->trans[s] : nullptr;
        io.invert[s] = s < d->S ? d->invert[s] : 0;
        io.grot[s] = s < d->S ? d->grad_rot[s] : nullptr;
        io.gtrans[s] = s < d->S ? d->grad_trans[s] : nullptr;
    }
}

// scratch of the intrinsics gradients in the ctx workspace of the current bank: arrival counter (16 bytes, zeroed when the
// slot is allocated; the reducing thread leaves it at 0) | (S*N, 18) doubles.  All null when no intrinsics gradient is asked.
static int intrinsics_io(md2_ctx* ctx, const md2_vsl_desc* d, IntrIO& k, cudaStream_t st) {
    memset(&k, 0, sizeof(k));
    if (!d->grad_K && !d->grad_invK) return 0;
    const int64_t gen = ctx->ws_gen[ctx->bank];
    char* buf = (char*)ws_get(ctx, MD2_WS_KGRAD, 16 + sizeof(double) * 18 * (size_t)d->S * d->N);
    if (!buf) return 1;
    if (ctx->ws_gen[ctx->bank] != gen) MD2_CHECK(cudaMemsetAsync(buf, 0, 16, st));
    k.gK = d->grad_K; k.giK = d->grad_invK;
    k.count = reinterpret_cast<unsigned*>(buf);
    k.part = reinterpret_cast<double*>(buf + 16);
    return 0;
}

enum { MODE_FWD = 0, MODE_BWD = 1, MODE_FWDBWD = 2 };

int run_vsl(md2_ctx* ctx, const md2_vsl_desc* d, int mode, float gloss, cudaStream_t st) {
    if (check_desc(d, true)) return 1;
    MD2_USE_DEVICE(ctx);
    const int W = d->W, H = d->H, N = d->N, L = d->L, S = d->S, C = d->C;
    const bool bwd = mode != MODE_FWD;

    FusedParams p;
    memset(&p, 0, sizeof(p));
    p.W = W; p.H = H; p.N = N; p.L = L; p.S = S;
    p.tgt = d->target; p.tgt_ns = d->target_image_stride;
    for (int s = 0; s < S; ++s) {
        p.src[s] = d->source[s]; p.src_ns[s] = d->source_image_stride[s];
        p.gsrc[s] = bwd ? d->grad_source[s] : nullptr;
        p.viz_warped[s] = d->viz_warped[s];
    }
    p.viz_loss = d->viz_loss;
    p.automask = d->automask;
    if (!d->automask && d->compute_automask) {
        // the automask pre-pass of the training loop (src/Monodepth.jl:159-164) as the first launch of this call
        float* am = (float*)ws_get(ctx, MD2_WS_AUTOMASK, sizeof(float) * (size_t)N * W * H);
        if (!am) return 1;
        int64_t ns[MAX_S];
        for (int s = 0; s < S; ++s) ns[s] = d->source_image_stride[s];
        if (launch_automask(ctx, S, d->source, ns, d->target, d->target_image_stride, am, W, H, C, N, st)) return 1;
        p.automask = am;
    }
    p.dbg = (bwd && !use_march_v1()) ? d->debug_choices : nullptr;
    if (d->debug_choices) MD2_REQUIRE(p.dbg != nullptr, "debug_choices is served by the value + gradient calls only");
    {   // the reference rounds min_disp and max_disp to T first (src/utils.jl:176-178)
        const float mind = (float)(1.0 / (double)d->max_depth), maxd = (float)(1.0 / (double)d->min_depth);
        p.depth_a = maxd - mind; p.depth_b = mind;
    }
    int n_low = 0, low_rows = 0;
    for (int l = 0; l < L; ++l) {
        p.smooth_w[l] = d->smooth_weight[l];
        p.disp[l] = d->disparity[l]; p.dw[l] = d->disp_w[l]; p.dh[l] = d->disp_h[l];
        p.usx[l] = up_scale(d->disp_w[l], W); p.usy[l] = up_scale(d->disp_h[l], H);
        p.gdisp[l] = bwd ? d->grad_disparity[l] : nullptr;
        if (bwd) MD2_REQUIRE(d->grad_disparity[l] != nullptr, "null grad_disparity");
        if (d->disp_w[l] != W || d->disp_h[l] != H) {
            ++n_low;
            low_rows += d->disp_h[l];
        }
    }
    if (n_low && taps_get(ctx, d, p, st)) return 1;
    {   // full-resolution views of every scale: the caller's buffers for native-size scales, L2-resident
        // scratch (upsampled disparity; full-resolution gradient before its adjoint down-sampling) otherwise
        const size_t img = (size_t)N * W * H;
        float* dscr = n_low ? (float*)ws_get(ctx, MD2_WS_DISP, sizeof(float) * img * n_low) : nullptr;
        float* gscr = (n_low && bwd) ? (float*)ws_get(ctx, MD2_WS_GDISP, sizeof(float) * img * n_low) : nullptr;
        if (n_low && (!dscr || (bwd && !gscr))) return 1;
        int k = 0;
        for (int l = 0; l < L; ++l) {
            const bool native = d->disp_w[l] == W && d->disp_h[l] == H;
            p.dfull[l] = native ? d->disparity[l] : dscr + img * k;
            p.gfull[l] = !bwd ? nullptr : (native ? d->grad_disparity[l] : gscr + img * k);
            if (!native) ++k;
        }
    }
    p.loss_scale = d->loss_scale;
    p.gloss = gloss;
    p.normalize_disp = d->normalize_disparity;
    p.mode = mode;
    fill_pose_io(d, p.pose);

    const bool v2 = !use_march_v1();   // the single-warp kernels (md2_march2.cuh) serve every mode; MD2_MARCH_V1=1: the round-1 warp-pair kernels
    p.m_R = choose_march_rows(W, H, L * N, v2 || bwd, ctx->sm_count, v2 ? march2_resident_of(C, S, p.automask != nullptr, bwd) : march_resident_of(C, S, bwd), p.m_group);
    static const bool dbg_env = getenv("MD2_DEBUG") != nullptr, generic_env = getenv("MD2_PREP_GENERIC") != nullptr;
    if (dbg_env) fprintf(stderr, "[md2] chunk height %d, %d groups of short last chunks per (scale, image)\n", p.m_R, p.m_group);
    const int tiles = cdiv(W, (v2 || bwd) ? 28 : 30) * cdiv(H, p.m_R);   // work items per (scale, image)
    const int NP = NSTAT + 12 * S;
    p.pose_slot = 0;
    // prep kernel partition: 31-column x 4-row patches, one warp each, eight warps per block
    const int prep_strips = cdiv(W, PREP_COLS), prep_chunks = cdiv(H, PREP_ROWS);
    const int prep_nblk = cdiv((long long)prep_strips * prep_chunks, PREP_WARPS);
    const int do_stats = mode == MODE_FWDBWD;
    const bool zero_gs = bwd && d->zero_grad_source != 0;
    // slices of the source images per (source, image): L2 prefetch (value + gradient calls) and optional zero-fill
    const int aux_blocks = bwd ? max(1, min(64, cdiv((long long)C * W * H, 8192))) : 0;
    const int zero_blocks = zero_gs ? aux_blocks : -aux_blocks;
    float* pose_ab = (float*)ws_get(ctx, MD2_WS_POSE, sizeof(float) * 24 * S * N);
    float* partial = (float*)ws_get(ctx, MD2_WS_PARTIAL, sizeof(float) * (size_t)tiles * L * N * NP);
    float* stats = (float*)ws_get(ctx, MD2_WS_STATS, sizeof(float) * (size_t)L * N * NSTAT);
    float* part2 = (float*)ws_get(ctx, MD2_WS_MISC, sizeof(float) * (size_t)prep_nblk * L * N * 4);
    if (!pose_ab || !partial || !stats || !part2) return 1;
    p.pose_ab = pose_ab; p.pose_e = pose_ab + (size_t)12 * S * N; p.partial = partial;
    p.stats = stats; p.stats_out = stats; p.saved = (mode == MODE_BWD) ? nullptr : d->saved;
    if (mode == MODE_BWD && d->saved) p.stats = d->saved;   // else the ctx holds the last forward's statistics
    p.loss = (mode == MODE_BWD) ? nullptr : d->loss;
    p.prep_part = do_stats ? part2 : nullptr;
    p.prep_nblk = prep_nblk;
    IntrIO intr;
    memset(&intr, 0, sizeof(intr));
    if (bwd && intrinsics_io(ctx, d, intr, st)) return 1;

    cudaEvent_t evp0 = nullptr, evp3 = nullptr;   // profile mode 2: the step's first and last time stamp
    if (ctx->prof_on == 2) {
        while (ctx->prof_used + 4 > ctx->prof_ev.size()) {
            cudaEvent_t e;
            MD2_CHECK(cudaEventCreate(&e));
            ctx->prof_ev.push_back(e);
        }
        evp0 = ctx->prof_ev[ctx->prof_used + 2]; evp3 = ctx->prof_ev[ctx->prof_used + 3];
        MD2_CHECK(cudaEventRecord(evp0, st));
    }
    {   // prep: poses, upsampled low-res disparities (+ smoothness sums for the fused fwd+bwd, + zero-fill)
        const int nb = (do_stats || n_low) ? prep_nblk : 0;
        dim3 g(1 + nb + S * aux_blocks, N);
        // usual decoder layout (low-res scales first, one full-resolution scale last, fused fwd+bwd): the lean kernel
        // (the lean kernel always forms the smoothness sums; calls that do not want them -- forward-only, separate backward -- ignore its partials)
        bool usual = nb > 0 && L >= 1 && L <= 4 && n_low == L - 1 && d->disp_w[L - 1] == W && d->disp_h[L - 1] == H;
        if (generic_env) usual = false;
#define MD2_PREPF(CC, NL) prep_fast_kernel<CC, NL><<<g, 32 * PREP_WARPS, 0, st>>>(p, prep_strips, prep_chunks, nb, pose_ab, part2, zero_blocks)
#define MD2_PREP(CC, LL) prep_kernel<CC, LL><<<g, 32 * PREP_WARPS, 0, st>>>(p, prep_strips, prep_chunks, nb, do_stats, pose_ab, part2, zero_blocks)
        if (usual && C == 1)      { if (L == 1) MD2_PREPF(1, 0); else if (L == 2) MD2_PREPF(1, 1); else if (L == 3) MD2_PREPF(1, 2); else MD2_PREPF(1, 3); }
        else if (usual)           { if (L == 1) MD2_PREPF(3, 0); else if (L == 2) MD2_PREPF(3, 1); else if (L == 3) MD2_PREPF(3, 2); else MD2_PREPF(3, 3); }
        else if (C == 1) { if (L == 1) MD2_PREP(1, 1); else if (L <= 4) MD2_PREP(1, 4); else MD2_PREP(1, 8); }
        else        { if (L == 1) MD2_PREP(3, 1); else if (L <= 4) MD2_PREP(3, 4); else MD2_PREP(3, 8); }
#undef MD2_PREPF
#undef MD2_PREP
        MD2_LAUNCH_CHECK(ctx);
    }

    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    if (ctx->prof_on) {
        if (ctx->prof_used + 2 > ctx->prof_ev.size()) {
            for (int k = 0; k < 2; ++k) {
                cudaEvent_t e;
                MD2_CHECK(cudaEventCreate(&e));
                ctx->prof_ev.push_back(e);
            }
        }
        ev0 = ctx->prof_ev[ctx->prof_used]; ev1 = ctx->prof_ev[ctx->prof_used + 1];
        ctx->prof_used += ctx->prof_on == 2 ? 4 : 2;
        MD2_CHECK(cudaEventRecord(ev0, st));
    }
    if (v2) {
        // the optional visualisation outputs of train_loss (src/training.jl:34-37,71-74; every 50th step of the reference's
        // loop) are written by the forward-only kernel; the value + gradient kernel does not carry them
        const bool viz = d->viz_loss || d->viz_warped[0] || (S > 1 && d->viz_warped[S - 1]);
        if (!bwd || viz) { if (dispatch_march2(ctx, C, S, p, st, false)) return 1; }
        if (bwd) { if (dispatch_march2(ctx, C, S, p, st, true)) return 1; }
    }
    else if (bwd) { if (dispatch_march<true>(ctx, C, S, p, st)) return 1; }
    else     { if (dispatch_march<false>(ctx, C, S, p, st)) return 1; }
    if (ev1) MD2_CHECK(cudaEventRecord(ev1, st));
    {   // loss / statistics, pose gradients, adjoint of the upsample for the low-res decoder scales
        const int blocks = 1 + (bwd ? S * N + low_rows * N : 0);
        MD2_CHECK(launch_after(2, finish_kernel, dim3(blocks), dim3(FIN_THREADS), sizeof(float) * ((W + 3) & ~3), st, p, NP, tiles, bwd ? 1 : 0, low_rows, intr));
        MD2_LAUNCH_CHECK(ctx);
    }
    if (evp3) MD2_CHECK(cudaEventRecord(evp3, st));
    return 0;
}

// ------------------------------------------------------------------------------------------
// Replay cache of the device-pointer fused calls.  A training loop calls md2_view_synthesis_loss_* with the same
// descriptors again and again (the framework's allocator hands out the same buffers every step), and a call is three
// dependent launches whose host-side cost (~3 x 5 us + the bookkeeping above) is in the order of the kernels' run time.
// The second time a (descriptor, mode, seed) is seen its launches are captured into a CUDA graph on an internal
// stream; from then on the call is ONE cudaGraphLaunch on the caller's stream (same ordering semantics as the kernel
// launches it replaces).  Anything that changes what the launches would be -- any byte of the descriptor, the
// workspace generation -- is part of the key.  MD2_NO_REPLAY=1 turns it off.
// ------------------------------------------------------------------------------------------
struct ReplayEntry {
    md2_vsl_desc desc;
    int mode; float seed; int64_t ws_gen;
    uint64_t hash = 0;
    int seen = 0;
    cudaGraphExec_t exec = nullptr;
    int launches = 0;
    uint64_t last_use = 0;
};
struct ReplayCache {
    static constexpr int CAP = 64;
    ReplayEntry e[CAP];
    int used = 0;
    uint64_t tick = 0;
    cudaStream_t cap_stream = nullptr;
};

void replay_destroy(md2_ctx* ctx) {
    ReplayCache* rc = static_cast<ReplayCache*>(ctx->replay);
    if (!rc) return;
    for (int i = 0; i < rc->used; ++i)
        if (rc->e[i].exec) cudaGraphExecDestroy(rc->e[i].exec);
    if (rc->cap_stream) cudaStreamDestroy(rc->cap_stream);
    delete rc;
    ctx->replay = nullptr;
}

static int run_vsl_cached(md2_ctx* ctx, const md2_vsl_desc* d, int mode, float gloss, cudaStream_t st) {
    static const bool off = [] { const char* e = getenv("MD2_NO_REPLAY"); return e && atoi(e) != 0; }();
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (off || !d || ctx->prof_on || ctx->bank != 0 || d->debug_choices ||
        cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone)   // (already inside someone's capture)
        return run_vsl(ctx, d, mode, gloss, st);
    if (!ctx->replay) {
        ReplayCache* n = new ReplayCache();
        if (cudaStreamCreateWithFlags(&n->cap_stream, cudaStreamNonBlocking) != cudaSuccess) { delete n; cudaGetLastError(); return run_vsl(ctx, d, mode, gloss, st); }
        ctx->replay = n;
    }
    ReplayCache* rc = static_cast<ReplayCache*>(ctx->replay);
    ++rc->tick;
    uint64_t hash = 1469598103934665603ULL;          // FNV-1a over the descriptor's bytes (a cheap pre-filter for the memcmp)
    {
        const unsigned char* b = reinterpret_cast<const unsigned char*>(d);
        for (size_t i = 0; i < sizeof(*d); ++i) hash = (hash ^ b[i]) * 1099511628211ULL;
    }
    ReplayEntry* hit = nullptr;
    for (int i = 0; i < rc->used; ++i) {
        ReplayEntry& e = rc->e[i];
        if (e.hash == hash && e.mode == mode && e.seed == gloss && memcmp(&e.desc, d, sizeof(*d)) == 0) { hit = &e; break; }
    }
    if (hit && hit->ws_gen != ctx->ws_gen[0]) {      // a workspace was re-allocated since: the graph holds dead pointers
        if (hit->exec) { cudaGraphExecDestroy(hit->exec); hit->exec = nullptr; }
        hit->seen = 0;
    }
    if (!hit) {                                      // first sighting: remember it (evicting the least recently used), run eagerly
        ReplayEntry* slot = nullptr;
        if (rc->used < ReplayCache::CAP) slot = &rc->e[rc->used++];
        else {
            slot = &rc->e[0];
            for (int i = 1; i < rc->used; ++i) if (rc->e[i].last_use < slot->last_use) slot = &rc->e[i];
            if (slot->exec) { cudaGraphExecDestroy(slot->exec); slot->exec = nullptr; }
        }
        memcpy(&slot->desc, d, sizeof(*d));
        slot->mode = mode; slot->seed = gloss; slot->hash = hash; slot->seen = 0; slot->exec = nullptr;
        hit = slot;
    }
    hit->last_use = rc->tick;
    if (hit->exec) {
        MD2_USE_DEVICE(ctx);
        MD2_CHECK(cudaGraphLaunch(hit->exec, st));
        ctx->launches += hit->launches;
        return 0;
    }
    if (hit->seen++ == 0) {                          // eager run: validates, sizes the workspaces
        const int rcode = run_vsl(ctx, d, mode, gloss, st);
        hit->ws_gen = ctx->ws_gen[0];
        if (rcode) hit->seen = 0;
        return rcode;
    }
    {   // second sighting: capture on the internal stream, then replay on the caller's
        MD2_USE_DEVICE(ctx);
        cudaGraph_t graph = nullptr;
        const int64_t before = ctx->launches;
        if (cudaStreamBeginCapture(rc->cap_stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); return run_vsl(ctx, d, mode, gloss, st); }
        const int rcode = run_vsl(ctx, d, mode, gloss, rc->cap_stream);
        const cudaError_t ce = cudaStreamEndCapture(rc->cap_stream, &graph);
        const int n_launch = (int)(ctx->launches - before);
        ctx->launches = before;
        if (rcode || ce != cudaSuccess || !graph || hit->ws_gen != ctx->ws_gen[0]) {
            if (graph) cudaGraphDestroy(graph);
            cudaGetLastError();
            hit->seen = 0;
            return run_vsl(ctx, d, mode, gloss, st);
        }
        const cudaError_t ie = cudaGraphInstantiate(&hit->exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ie != cudaSuccess) { hit->exec = nullptr; cudaGetLastError(); hit->seen = 0; return run_vsl(ctx, d, mode, gloss, st); }
        hit->launches = n_launch;
        MD2_CHECK(cudaGraphLaunch(hit->exec, st));
        ctx->launches += hit->launches;
    }
    return 0;
}

// ------------------------------------------------------------------------------------------
// A15 `warp` (called at src/simple_depth.jl:30-32, body inferred from src/training.jl:48-57):
// disparity -> S warped images, thread per pixel, and its adjoint
// ------------------------------------------------------------------------------------------
struct WarpIO {
    float* out[MAX_S];          // fwd: (N,C,H,W) contiguous
    const float* gout[MAX_S];   // bwd
};

__global__ void pose_prep_kernel(PoseIO io, int S, int N, float* __restrict__ pose_ab) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= S * N) return;
    prepare_pose_one(io, i / N, i % N, pose_ab + (long long)i * 12);
}

__global__ void pose_final_kernel(PoseIO io, IntrIO intr, int S, int N, int NP, const float* __restrict__ sums) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= S * N) return;
    const int s = i / N, n = i % N;
    double G[9], h[3];
    const float* su = sums + (long long)n * NP + NSTAT + 12 * s;
    for (int k = 0; k < 9; ++k) G[k] = su[k];
    for (int k = 0; k < 3; ++k) h[k] = su[9 + k];
    finalize_pose(io, s, n, G, h);
    if (intr.part) {
        intrinsics_part(io, s, n, G, h, intr.part + 18 * (long long)i);
        if (intrinsics_last(intr, S, N)) {
            reduce_intrinsics(intr, io.kstride, S, N);
            *intr.count = 0u;
        }
    }
}

template <int C, int S>
__global__ void __launch_bounds__(256) warp_fwd_kernel(const __grid_constant__ FusedParams p, WarpIO io) {
    using F = Sampler<C>;
    const long long HW = (long long)p.W * p.H;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= HW * p.N) return;
    const int n = (int)(i / HW), pix = (int)(i % HW), gx = pix % p.W, gy = pix / p.W;
    const float d = p.disp[0][i];
#pragma unroll
    for (int s = 0; s < S; ++s) {
        typename F::Warped w; Taps tp; Proj pr;
        const float z = rcp_acc(fmaf(d, p.depth_a, p.depth_b));
        F::project_pixel(p, p.pose_ab + ((long long)s * p.N + n) * 12, gx, gy, z, pr, tp);
        F::template gather<false>(p, n, s, tp, w);
#pragma unroll
        for (int c = 0; c < C; ++c) io.out[s][((long long)n * C + c) * HW + pix] = w.val[c];
    }
}

template <int C, int S>
__global__ void __launch_bounds__(256) warp_bwd_kernel(const __grid_constant__ FusedParams p, WarpIO io) {
    using F = Sampler<C>;
    __shared__ float scratch[(NSTAT + 12 * S) * 8];
    const long long HW = (long long)p.W * p.H;
    const int n = blockIdx.y;
    constexpr int NP = NSTAT + 12 * S;
    float v[NP];
#pragma unroll
    for (int k = 0; k < NP; ++k) v[k] = 0.f;
    // (uniform trip count: every lane of a warp takes part in the shuffles of the merged scatter; lanes past the end idle)
    const int lane = threadIdx.x & 31;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long base = (long long)blockIdx.x * blockDim.x; base < HW; base += stride) {
        const long long pl = base + threadIdx.x;
        const bool active = pl < HW;
        const int pix = active ? (int)pl : 0, gx = pix % p.W, gy = pix / p.W;
        const float d = p.disp[0][(long long)n * HW + pix];
        float dbar_z = 0.f, zz = 0.f;
#pragma unroll
        for (int s = 0; s < S; ++s) {
            typename F::Warped w; float ibar[C]; Taps tp; Proj pr;
            const float z = rcp_acc(fmaf(d, p.depth_a, p.depth_b));
            F::project_pixel(p, p.pose_ab + ((long long)s * p.N + n) * 12, gx, gy, z, pr, tp);
            F::template gather<true>(p, n, s, tp, w);
            zz = z;
            float du = 0.f, dv = 0.f;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                ibar[c] = active ? io.gout[s][((long long)n * C + c) * HW + pix] : 0.f;
                du = fmaf(ibar[c], w.dix[c], du);
                dv = fmaf(ibar[c], w.diy[c], dv);
            }
            du *= tp.mx; dv *= tp.my;
            if (p.gsrc[s]) {   // (uniform: a launch parameter)
                float* gb = p.gsrc[s] + (long long)n * p.src_ns[s];
                const float w00 = (1.f - tp.fx) * (1.f - tp.fy), w01 = tp.fx * (1.f - tp.fy);
                const float w10 = (1.f - tp.fx) * tp.fy, w11 = tp.fx * tp.fy;
                const bool xr = tp.x0 + 1 < p.W, yb = tp.y0 + 1 < p.H;
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    float* r0 = gb + c * HW + (long long)tp.y0 * p.W + tp.x0;
                    float* r1 = r0 + p.W;
                    red_pair_merged(active ? r0 : nullptr, (active && xr) ? r0 + 1 : nullptr, w00 * ibar[c], w01 * ibar[c], lane);
                    red_pair_merged((active && yb) ? r1 : nullptr, (active && yb && xr) ? r1 + 1 : nullptr, w10 * ibar[c], w11 * ibar[c], lane);
                }
            }
            float cb[3];
            project_ab_bwd(pr, du, dv, cb);
            dbar_z += cb[0] * pr.ap[0] + cb[1] * pr.ap[1] + cb[2] * pr.ap[2];
            const float zp[3] = {z * (float)(gx + 1), z * (float)(gy + 1), z};
#pragma unroll
            for (int a = 0; a < 3; ++a) {
#pragma unroll
                for (int b = 0; b < 3; ++b) v[NSTAT + 12 * s + 3 * a + b] = fmaf(cb[a], zp[b], v[NSTAT + 12 * s + 3 * a + b]);
                v[NSTAT + 12 * s + 9 + a] += cb[a];
            }
        }
        if (active) p.gdisp[0][(long long)n * HW + pix] = -p.depth_a * zz * zz * dbar_z;
    }
    block_sum<NP>(v, scratch);
    if (threadIdx.x < NP)
        p.partial[((long long)n * gridDim.x + blockIdx.x) * NP + threadIdx.x] = scratch[threadIdx.x * (blockDim.x >> 5)];
}

static int run_warp(md2_ctx* ctx, const md2_vsl_desc* d, float* const* out, const float* const* gout, cudaStream_t st) {
    if (check_desc(d, false)) return 1;
    MD2_USE_DEVICE(ctx);
    const int W = d->W, H = d->H, N = d->N, S = d->S, C = d->C;
    const long long HW = (long long)W * H;
    const bool bwd = gout != nullptr;
    MD2_REQUIRE(d->disparity[0] != nullptr, "null disparity");
    MD2_REQUIRE(d->disp_w[0] == W && d->disp_h[0] == H, "warp needs a full-resolution disparity");
    FusedParams p;
    memset(&p, 0, sizeof(p));
    p.W = W; p.H = H; p.N = N; p.L = 1; p.S = S;
    WarpIO io;
    memset(&io, 0, sizeof(io));
    for (int s = 0; s < S; ++s) {
        p.src[s] = d->source[s]; p.src_ns[s] = d->source_image_stride[s];
        p.gsrc[s] = bwd ? d->grad_source[s] : nullptr;
        if (bwd) { MD2_REQUIRE(gout[s] != nullptr, "null upstream gradient"); io.gout[s] = gout[s]; }
        else { MD2_REQUIRE(out && out[s], "null output"); io.out[s] = out[s]; }
    }
    const float mind = (float)(1.0 / (double)d->max_depth), maxd = (float)(1.0 / (double)d->min_depth);
    p.depth_a = maxd - mind; p.depth_b = mind;
    p.disp[0] = d->disparity[0]; p.dw[0] = W; p.dh[0] = H;
    fill_pose_io(d, p.pose);
    float* pose_ab = (float*)ws_get(ctx, MD2_WS_POSE, sizeof(float) * 12 * S * N);
    if (!pose_ab) return 1;
    pose_prep_kernel<<<cdiv(S * N, 64), 64, 0, st>>>(p.pose, S, N, pose_ab);
    MD2_LAUNCH_CHECK(ctx);
    p.pose_ab = pose_ab;
    if (!bwd) {
        const int g = cdiv(HW * N, 256);
        if (C == 1 && S == 1) warp_fwd_kernel<1, 1><<<g, 256, 0, st>>>(p, io);
        else if (C == 1 && S == 2) warp_fwd_kernel<1, 2><<<g, 256, 0, st>>>(p, io);
        else if (C == 3 && S == 1) warp_fwd_kernel<3, 1><<<g, 256, 0, st>>>(p, io);
        else warp_fwd_kernel<3, 2><<<g, 256, 0, st>>>(p, io);
        MD2_LAUNCH_CHECK(ctx);
        return 0;
    }
    MD2_REQUIRE(d->grad_disparity[0] != nullptr, "null grad_disparity");
    p.gdisp[0] = d->grad_disparity[0];
    const int NP = NSTAT + 12 * S;
    const int bpi = max(1, min(128, cdiv(HW, 1024)));
    float* partial = (float*)ws_get(ctx, MD2_WS_PARTIAL, sizeof(float) * (size_t)bpi * N * NP);
    float* sums = (float*)ws_get(ctx, MD2_WS_SUMS, sizeof(float) * (size_t)N * NP);
    if (!partial || !sums) return 1;
    p.partial = partial;
    dim3 g(bpi, N);
    if (C == 1 && S == 1) warp_bwd_kernel<1, 1><<<g, 256, 0, st>>>(p, io);
    else if (C == 1 && S == 2) warp_bwd_kernel<1, 2><<<g, 256, 0, st>>>(p, io);
    else if (C == 3 && S == 1) warp_bwd_kernel<3, 1><<<g, 256, 0, st>>>(p, io);
    else warp_bwd_kernel<3, 2><<<g, 256, 0, st>>>(p, io);
    MD2_LAUNCH_CHECK(ctx);
    if (launch_reduce_partials(ctx, partial, sums, NP, nullptr, N, bpi, NP, st)) return 1;
    IntrIO intr;
    if (intrinsics_io(ctx, d, intr, st)) return 1;
    pose_final_kernel<<<cdiv(S * N, 64), 64, 0, st>>>(p.pose, intr, S, N, NP, sums);
    MD2_LAUNCH_CHECK(ctx);
    return 0;
}

}  // namespace md2

// ------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------
extern "C" {

const char* md2_version(void) { return "md2_b200 0.1.0 (sm_100a)"; }
const char* md2_last_error(void) { return md2::last_error_ref().c_str(); }

int md2_create(int device, md2_ctx** out) {
    if (!out) return md2::set_error("md2_create: null out pointer");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return md2::set_error("md2_create: no CUDA device (%s); this library has no CPU fallback",
                              cudaGetErrorString(e));
    if (device < 0 || device >= count) return md2::set_error("md2_create: bad device %d", device);
    md2_ctx* c = new md2_ctx();
    c->device = device;
    c->launches = 0;
    c->sm_count = 148;
    cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
    *out = c;
    return 0;
}

int md2_destroy(md2_ctx* ctx) {
    if (!ctx) return 0;
    md2::DeviceGuard guard(ctx->device);
    cudaDeviceSynchronize();
    for (int b = 0; b < MD2_WS_BANKS; ++b)
        for (int i = 0; i < MD2_WS_COUNT; ++i)
            if (ctx->ws[b][i].ptr) cudaFree(ctx->ws[b][i].ptr);
    for (cudaEvent_t e : ctx->prof_ev) cudaEventDestroy(e);
    md2::host_path_destroy(ctx);
    md2::opt_path_destroy(ctx);
    md2::replay_destroy(ctx);
    md2::taps_destroy(ctx);
    delete ctx;
    return 0;
}

int64_t md2_launch_count(const md2_ctx* ctx) { return ctx ? ctx->launches : 0; }

int md2_profile_enable(md2_ctx* ctx, int32_t on) {
    MD2_REQUIRE(ctx != nullptr, "null ctx");
    ctx->prof_on = on;
    ctx->prof_used = 0;
    return 0;
}
int md2_profile_read(md2_ctx* ctx, float* total_ms, int64_t* launches) {
    MD2_REQUIRE(ctx != nullptr && total_ms && launches, "bad arguments");
    const size_t per = ctx->prof_on == 2 ? 4 : 2;
    float tot = 0.f;
    for (size_t i = 0; i + per <= ctx->prof_used; i += per) {
        MD2_CHECK(cudaEventSynchronize(ctx->prof_ev[i + 1]));
        float ms = 0.f;
        MD2_CHECK(cudaEventElapsedTime(&ms, ctx->prof_ev[i], ctx->prof_ev[i + 1]));
        tot += ms;
    }
    *total_ms = tot;
    *launches = (int64_t)(ctx->prof_used / per);
    ctx->prof_used = 0;
    return 0;
}
int md2_profile_read_phases(md2_ctx* ctx, float* prep_ms, float* march_ms, float* finish_ms, int64_t* launches) {
    MD2_REQUIRE(ctx != nullptr && prep_ms && march_ms && finish_ms && launches, "bad arguments");
    MD2_REQUIRE(ctx->prof_on == 2, "md2_profile_enable(ctx, 2) first");
    float a = 0.f, b = 0.f, c = 0.f;
    for (size_t i = 0; i + 4 <= ctx->prof_used; i += 4) {
        MD2_CHECK(cudaEventSynchronize(ctx->prof_ev[i + 3]));
        float ms = 0.f;
        MD2_CHECK(cudaEventElapsedTime(&ms, ctx->prof_ev[i + 2], ctx->prof_ev[i])); a += ms;       // prep
        MD2_CHECK(cudaEventElapsedTime(&ms, ctx->prof_ev[i], ctx->prof_ev[i + 1])); b += ms;       // march
        MD2_CHECK(cudaEventElapsedTime(&ms, ctx->prof_ev[i + 1], ctx->prof_ev[i + 3])); c += ms;   // finish
    }
    *prep_ms = a; *march_ms = b; *finish_ms = c;
    *launches = (int64_t)(ctx->prof_used / 4);
    ctx->prof_used = 0;
    return 0;
}

int md2_view_synthesis_loss_fwd(md2_ctx* ctx, const md2_vsl_desc* d, md2_stream st) {
    MD2_REQUIRE(ctx != nullptr, "null ctx");
    return md2::run_vsl_cached(ctx, d, md2::MODE_FWD, 0.f, (cudaStream_t)st);
}
int md2_view_synthesis_loss_bwd(md2_ctx* ctx, const md2_vsl_desc* d, float upstream, md2_stream st) {
    MD2_REQUIRE(ctx != nullptr, "null ctx");
    return md2::run_vsl_cached(ctx, d, md2::MODE_BWD, upstream, (cudaStream_t)st);
}
int md2_view_synthesis_loss_fwdbwd(md2_ctx* ctx, const md2_vsl_desc* d, float seed, md2_stream st) {
    MD2_REQUIRE(ctx != nullptr, "null ctx");
    return md2::run_vsl_cached(ctx, d, md2::MODE_FWDBWD, seed, (cudaStream_t)st);
}

int md2_warp_fwd(md2_ctx* ctx, const md2_vsl_desc* d, float* const* out, md2_stream st) {
    MD2_REQUIRE(ctx != nullptr, "null ctx");
    return md2::run_warp(ctx, d, out, nullptr, (cudaStream_t)st);
}
int md2_warp_bwd(md2_ctx* ctx, const md2_vsl_desc* d, const float* const* gout, md2_stream st) {
    MD2_REQUIRE(ctx != nullptr, "null ctx");
    MD2_REQUIRE(gout != nullptr, "null upstream gradients");
    return md2::run_warp(ctx, d, nullptr, gout, (cudaStream_t)st);
}

int md2_upsample_bilinear_fwd(md2_ctx* ctx, const float* in, float* out, int32_t w, int32_t h, int32_t W, int32_t H,
                              int32_t CN, md2_stream st) {
    MD2_REQUIRE(ctx != nullptr, "null ctx");
    MD2_USE_DEVICE(ctx);
    MD2_REQUIRE(in && out && w > 0 && h > 0 && W > 0 && H > 0 && CN > 0, "bad arguments");
    md2::upsample_kernel<<<md2::cdiv((long long)W * H * CN, 256), 256, 0, (cudaStream_t)st>>>(in, out, w, h, W, H, CN);
    MD2_LAUNCH_CHECK(ctx);
    return 0;
}
int md2_upsample_bilinear_bwd(md2_ctx* ctx, const float* gout, float* gin, int32_t w, int32_t h, int32_t W, int32_t H,
                              int32_t CN, md2_stream st) {
    MD2_REQUIRE(ctx != nullptr, "null ctx");
    MD2_USE_DEVICE(ctx);
    MD2_REQUIRE(gout && gin && w > 0 && h > 0 && W > 0 && H > 0 && CN > 0, "bad arguments");
    md2::upsample_bwd_kernel<<<md2::cdiv((long long)w * h * CN, 128), 128, 0, (cudaStream_t)st>>>(gout, gin, w, h, W, H, CN);
    MD2_LAUNCH_CHECK(ctx);
    return 0;
}

}  // extern "C"
