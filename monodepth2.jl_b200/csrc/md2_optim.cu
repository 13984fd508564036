// Optimiser side of the loss path: the Flux ADAM update as one multi-tensor kernel (md2_adam_step) and the reference's
// single-triplet optimiser `slow_depth` (src/simple_depth.jl:1-62) as a device-resident loop (md2_slow_depth): one
// iteration = fused value + gradient of the objective (three launches, md2_fused.cu) + one ADAM launch, captured once
// into a CUDA graph and replayed, so 500 iterations cost 500 graph launches and no host round trip.
#include <string.h>

#include "md2_common.cuh"
#include "md2_fused.cuh"

namespace md2 {

int run_vsl(md2_ctx* ctx, const md2_vsl_desc* d, int mode, float gloss, cudaStream_t st);   // md2_fused.cu

struct AdamArgs {
    float* p[MD2_ADAM_MAX_TENSORS];
    const float* g[MD2_ADAM_MAX_TENSORS];
    long long off[MD2_ADAM_MAX_TENSORS + 1];   // prefix sums of the element counts (state = [m | v] of the concatenation)
    int n;
    int vec4;                                  // every tensor 16-byte aligned with a count that is a multiple of 4
};

// Flux.Optimise.ADAM (Flux optimisers.jl, apply!):  m = b1 m + (1-b1) g;  v = b2 v + (1-b2) g^2;
//   p -= lr * m / (1 - b1^t) / (sqrt(v / (1 - b2^t)) + eps),  t = 1, 2, ...
// clock[0] = number of updates applied so far (device-resident, so that a captured graph advances it by itself),
// clock[1] = arrival counter of the blocks of one launch: the last block to arrive publishes t and resets it -- every
// block has read clock[0] before it arrives, so no block ever sees the incremented value of its own launch.
template <bool VEC4>
__global__ void __launch_bounds__(256) adam_kernel(const __grid_constant__ AdamArgs a, float* __restrict__ state,
                                                   unsigned long long* __restrict__ clock, float lr, float b1, float b2, float eps,
                                                   float gscale, const float* __restrict__ loss_in, float* __restrict__ history,
                                                   long long history_len) {
    const unsigned long long t0 = *reinterpret_cast<volatile unsigned long long*>(clock);
    const double t = (double)(t0 + 1);
    const float c1 = (float)(1.0 / (1.0 - pow((double)b1, t)));
    const float c2 = (float)(1.0 / (1.0 - pow((double)b2, t)));
    const long long total = a.off[a.n];
    float* __restrict__ mm = state;
    float* __restrict__ vv = state + total;
    const long long stride = (long long)gridDim.x * blockDim.x * (VEC4 ? 4 : 1);
    for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * (VEC4 ? 4 : 1); i < total; i += stride) {
        int k = 0;
#pragma unroll 1
        while (k + 1 < a.n && i >= a.off[k + 1]) ++k;
        const long long j = i - a.off[k];
        if (VEC4) {
            float4 g = __ldcs(reinterpret_cast<const float4*>(a.g[k] + j));
            float4 p = *reinterpret_cast<const float4*>(a.p[k] + j);
            float4 m = *reinterpret_cast<const float4*>(mm + i);
            float4 v = *reinterpret_cast<const float4*>(vv + i);
#define MD2_ADAM1(c)                                                    \
    {                                                                   \
        const float gg = g.c * gscale;                                  \
        m.c = fmaf(b1, m.c, (1.0f - b1) * gg);                          \
        v.c = fmaf(b2, v.c, (1.0f - b2) * gg * gg);                     \
        p.c -= lr * (m.c * c1) / (sqrtf(v.c * c2) + eps);               \
    }
            MD2_ADAM1(x) MD2_ADAM1(y) MD2_ADAM1(z) MD2_ADAM1(w)
#undef MD2_ADAM1
            *reinterpret_cast<float4*>(a.p[k] + j) = p;
            *reinterpret_cast<float4*>(mm + i) = m;
            *reinterpret_cast<float4*>(vv + i) = v;
        } else {
            const float gg = a.g[k][j] * gscale;
            const float m = fmaf(b1, mm[i], (1.0f - b1) * gg);
            const float v = fmaf(b2, vv[i], (1.0f - b2) * gg * gg);
            mm[i] = m; vv[i] = v;
            a.p[k][j] -= lr * (m * c1) / (sqrtf(v * c2) + eps);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned long long arrived = atomicAdd(clock + 1, 1ULL);
        if (arrived == gridDim.x - 1) {
            if (history && (long long)t0 < history_len) history[t0] = *loss_in;
            clock[1] = 0ULL;
            __threadfence();
            *reinterpret_cast<volatile unsigned long long*>(clock) = t0 + 1;
        }
    }
}

static int launch_adam(md2_ctx* ctx, int n, float* const* params, const float* const* grads, const int64_t* counts, float* state,
                       int64_t* clock, float lr, float b1, float b2, float eps, float gscale, const float* loss_in, float* history,
                       int64_t history_len, cudaStream_t st) {
    MD2_REQUIRE(n >= 1 && n <= MD2_ADAM_MAX_TENSORS, "1 .. MD2_ADAM_MAX_TENSORS tensors per call");
    MD2_REQUIRE(params && grads && counts && state && clock, "null argument");
    AdamArgs a;
    memset(&a, 0, sizeof(a));
    a.n = n; a.vec4 = 1;
    long long off = 0;
    for (int k = 0; k < n; ++k) {
        MD2_REQUIRE(params[k] && grads[k] && counts[k] > 0, "null tensor / empty tensor");
        a.p[k] = params[k]; a.g[k] = grads[k]; a.off[k] = off;
        off += counts[k];
        if ((counts[k] & 3) || (reinterpret_cast<uintptr_t>(params[k]) & 15) || (reinterpret_cast<uintptr_t>(grads[k]) & 15)) a.vec4 = 0;
    }
    a.off[n] = off;
    if ((reinterpret_cast<uintptr_t>(state) & 15) || (off & 3)) a.vec4 = 0;
    const long long work = a.vec4 ? off / 4 : off;
    long long blocks = (work + 255) / 256;
    const long long cap = (long long)ctx->sm_count * 8;    // grid-stride beyond one resident wave
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    unsigned long long* ck = reinterpret_cast<unsigned long long*>(clock);
    if (a.vec4) adam_kernel<true><<<(int)blocks, 256, 0, st>>>(a, state, ck, lr, b1, b2, eps, gscale, loss_in, history, history_len);
    else adam_kernel<false><<<(int)blocks, 256, 0, st>>>(a, state, ck, lr, b1, b2, eps, gscale, loss_in, history, history_len);
    MD2_LAUNCH_CHECK(ctx);
    return 0;
}

// ---- slow_depth ------------------------------------------------------------------------------------------------
struct OptPath {
    cudaStream_t st = nullptr;
    cudaEvent_t ev_in = nullptr, ev_out = nullptr;
    cudaGraphExec_t exec = nullptr;
    md2_vsl_desc key;
    float key_hp[4] = {0, 0, 0, 0};
    const void* key_ptrs[4] = {nullptr, nullptr, nullptr, nullptr};
    int64_t key_len = 0, key_ws_gen = -1;
    bool have_key = false;
};

static OptPath* opt_path(md2_ctx* ctx) {
    if (!ctx->opt) {
        OptPath* o = new OptPath();
        const bool ok = cudaStreamCreateWithFlags(&o->st, cudaStreamNonBlocking) == cudaSuccess &&
                        cudaEventCreateWithFlags(&o->ev_in, cudaEventDisableTiming) == cudaSuccess &&
                        cudaEventCreateWithFlags(&o->ev_out, cudaEventDisableTiming) == cudaSuccess;
        if (!ok) {
            set_error("slow_depth: stream / event creation failed: %s", cudaGetErrorString(cudaGetLastError()));
            delete o;
            return nullptr;
        }
        ctx->opt = o;
    }
    return static_cast<OptPath*>(ctx->opt);
}

void opt_path_destroy(md2_ctx* ctx) {
    OptPath* o = static_cast<OptPath*>(ctx->opt);
    if (!o) return;
    if (o->exec) cudaGraphExecDestroy(o->exec);
    cudaStreamDestroy(o->st);
    cudaEventDestroy(o->ev_in); cudaEventDestroy(o->ev_out);
    delete o;
    ctx->opt = nullptr;
}

// one iteration on stream st: value + gradient of the objective, then ADAM on (disparity, rvec_s, tvec_s)
static int slow_depth_iteration(md2_ctx* ctx, const md2_vsl_desc* d, float lr, float b1, float b2, float eps, float* state, int64_t* clock,
                                float* history, int64_t history_len, cudaStream_t st) {
    if (run_vsl(ctx, d, /*MODE_FWDBWD*/ 2, 1.0f, st)) return 1;
    float* params[MD2_ADAM_MAX_TENSORS];
    const float* grads[MD2_ADAM_MAX_TENSORS];
    int64_t counts[MD2_ADAM_MAX_TENSORS];
    int n = 0;
    params[n] = const_cast<float*>(d->disparity[0]); grads[n] = d->grad_disparity[0]; counts[n++] = (int64_t)d->W * d->H * d->N;
    for (int s = 0; s < d->S; ++s) {
        params[n] = const_cast<float*>(d->rot[s]); grads[n] = d->grad_rot[s]; counts[n++] = 3LL * d->N;
        params[n] = const_cast<float*>(d->trans[s]); grads[n] = d->grad_trans[s]; counts[n++] = 3LL * d->N;
    }
    return launch_adam(ctx, n, params, grads, counts, state, clock, lr, b1, b2, eps, 1.0f, d->loss, history, history_len, st);
}

static int run_slow_depth(md2_ctx* ctx, const md2_vsl_desc* d, int iters, float lr, float b1, float b2, float eps, float* state,
                          int64_t* clock, float* history, int64_t history_len, cudaStream_t caller) {
    MD2_REQUIRE(d != nullptr && state && clock, "null argument");
    MD2_REQUIRE(iters >= 0, "iters must be >= 0");
    MD2_REQUIRE(d->L == 1 && d->disp_w[0] == d->W && d->disp_h[0] == d->H, "one full-resolution disparity (src/simple_depth.jl:8)");
    MD2_REQUIRE(d->pose_mode == 1, "poses are (rvec, tvec) parameters: pose_mode must be 1");
    MD2_REQUIRE(!d->grad_K && !d->grad_invK, "grad_K / grad_invK must be NULL: the intrinsics are not among the optimised tensors");
    MD2_REQUIRE(d->per_image_K == 0 || d->per_image_K == 1, "per_image_K must be 0 or 1");
    MD2_REQUIRE(d->loss && d->grad_disparity[0], "loss / grad_disparity scratch is required");
    for (int s = 0; s < d->S; ++s) MD2_REQUIRE(d->grad_rot[s] && d->grad_trans[s], "grad_rot / grad_trans scratch is required");
    MD2_REQUIRE(!d->debug_choices && !d->saved && !d->viz_loss && !d->viz_warped[0] && !d->viz_warped[1], "debug / saved / viz outputs are not served here");
    if (iters == 0) return 0;
    MD2_USE_DEVICE(ctx);
    MD2_REQUIRE(!ctx->prof_on, "kernel profiling (md2_profile_enable) is not available inside md2_slow_depth");
    OptPath* o = opt_path(ctx);
    if (!o) return 1;
    // the loop runs on an internal stream (the caller's may be the legacy default stream, which cannot be captured),
    // ordered after everything the caller has enqueued so far and before everything it enqueues afterwards
    MD2_CHECK(cudaEventRecord(o->ev_in, caller));
    MD2_CHECK(cudaStreamWaitEvent(o->st, o->ev_in, 0));
    const float hp[4] = {lr, b1, b2, eps};
    const void* ptrs[4] = {state, clock, history, nullptr};
    int done = 0;
    const bool same = o->have_key && o->exec && o->key_ws_gen == ctx->ws_gen[0] && o->key_len == history_len &&
                      memcmp(&o->key, d, sizeof(*d)) == 0 && memcmp(o->key_hp, hp, sizeof(hp)) == 0 && memcmp(o->key_ptrs, ptrs, sizeof(ptrs)) == 0;
    if (!same) {
        if (o->exec) { cudaGraphExecDestroy(o->exec); o->exec = nullptr; }
        o->have_key = false;
        // first iteration eagerly: validates the descriptor and sizes every workspace (no allocation under capture)
        if (slow_depth_iteration(ctx, d, lr, b1, b2, eps, state, clock, history, history_len, o->st)) return 1;
        done = 1;
        if (iters > 1 && !getenv("MD2_OPT_NO_GRAPH")) {
            cudaGraph_t graph = nullptr;
            const int64_t launches = ctx->launches;
            MD2_CHECK(cudaStreamBeginCapture(o->st, cudaStreamCaptureModeThreadLocal));
            const int rc = slow_depth_iteration(ctx, d, lr, b1, b2, eps, state, clock, history, history_len, o->st);
            const cudaError_t ce = cudaStreamEndCapture(o->st, &graph);
            ctx->launches = launches;
            if (rc || ce != cudaSuccess || !graph) {
                if (graph) cudaGraphDestroy(graph);
                cudaGetLastError();
                if (rc) return 1;
                return set_error("slow_depth: stream capture failed: %s", cudaGetErrorString(ce));
            }
            const cudaError_t ie = cudaGraphInstantiate(&o->exec, graph, 0);
            cudaGraphDestroy(graph);
            if (ie != cudaSuccess) { o->exec = nullptr; return set_error("slow_depth: cudaGraphInstantiate failed: %s", cudaGetErrorString(ie)); }
            memcpy(&o->key, d, sizeof(*d)); memcpy(o->key_hp, hp, sizeof(hp)); memcpy(o->key_ptrs, ptrs, sizeof(ptrs));
            o->key_len = history_len; o->key_ws_gen = ctx->ws_gen[0]; o->have_key = true;
        }
    }
    for (; done < iters; ++done) {
        if (o->exec) {
            MD2_CHECK(cudaGraphLaunch(o->exec, o->st));
            ctx->launches += 4;
        } else if (slow_depth_iteration(ctx, d, lr, b1, b2, eps, state, clock, history, history_len, o->st)) return 1;
    }
    MD2_CHECK(cudaEventRecord(o->ev_out, o->st));
    MD2_CHECK(cudaStreamWaitEvent(caller, o->ev_out, 0));
    return 0;
}

}  // namespace md2

extern "C" {

int md2_adam_step(md2_ctx* ctx, int32_t n, float* const* params, const float* const* grads, const int64_t* counts, float* state,
                  int64_t* clock, float lr, float beta1, float beta2, float eps, float grad_scale, md2_stream st) {
    MD2_REQUIRE(ctx != nullptr, "null ctx");
    MD2_USE_DEVICE(ctx);
    return md2::launch_adam(ctx, n, params, grads, counts, state, clock, lr, beta1, beta2, eps, grad_scale, nullptr, nullptr, 0, (cudaStream_t)st);
}

int md2_slow_depth(md2_ctx* ctx, const md2_vsl_desc* d, int32_t iters, float lr, float beta1, float beta2, float eps, float* state,
                   int64_t* clock, float* loss_history, int64_t history_len, md2_stream st) {
    MD2_REQUIRE(ctx != nullptr, "null ctx");
    return md2::run_slow_depth(ctx, d, iters, lr, beta1, beta2, eps, state, clock, loss_history, history_len, (cudaStream_t)st);
}

}  // extern "C"
