/* md2.h -- C ABI of libmd2_b200.so: hand-written sm_100a CUDA kernels for the
 * view-synthesis loss path of pxl-th/Monodepth2.jl (warp + SSIM/L1 photometric loss,
 * forward and backward).  This is the drop-in boundary: Julia binds it with `ccall`
 * (INTEGRATION.md, monodepth2.jl_b200/julia/Monodepth2B200.jl), the tests and bench bind it
 * with Python ctypes.
 *
 * The reference has no FFI of its own: each entry point below replaces a plain Julia
 * function (plus its Zygote/ChainRules pullback) and cites it as file:line in
 * /root/reference (= pxl-th/Monodepth2.jl).
 *
 * Conventions
 *  - every function returns 0 on success, non-zero on error; the message is available
 *    through md2_last_error() (thread-local).  Nothing throws or exits.
 *  - every tensor argument is a caller-owned DEVICE pointer to contiguous float32 in
 *    Julia (column-major) memory order: image (W,H,C,N), disparity (W,H,1,N), points
 *    (3,P,N) with p = (h-1)W + (w-1), grid (2,W,H,N), K/invK (3,3) (or (3,3,N): md2_vsl_desc.per_image_K), R (3,3,N), t (3,1,N),
 *    rvec (3,N).  (W,H,C,N) column-major is bit-identical to row-major NCHW.
 *  - pixel coordinates are 1-based like the reference (src/utils.jl:47-51); frame indices
 *    passed through this ABI are 0-based.
 *  - calls are asynchronous on `stream` (a cudaStream_t passed as void*; NULL = legacy
 *    default stream) and never synchronise the device.  Scratch lives in the md2_ctx
 *    (one per device and host thread; not thread-safe; grown on demand, which may call
 *    cudaMalloc on first use of a larger shape).
 *  - gradient outputs are overwritten unless documented as "accumulated".
 */
#ifndef MD2_H
#define MD2_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MD2_MAX_SOURCES 2
#define MD2_MAX_SCALES 8
#define MD2_ADAM_MAX_TENSORS 16
#define MD2_HOST_LANES 3

typedef struct md2_ctx md2_ctx;
typedef void* md2_stream;

const char* md2_version(void);
const char* md2_last_error(void);
int md2_create(int device, md2_ctx** out);
int md2_destroy(md2_ctx* ctx);
/* number of kernels launched through this ctx since creation (bench's gpu_launches) */
int64_t md2_launch_count(const md2_ctx* ctx);
/* device-side timing of the dominant kernel (the marching kernel of
 * md2_view_synthesis_loss_*): while enabled, every such launch is bracketed by CUDA events on
 * the launch stream; md2_profile_read waits for them, returns the summed duration and the
 * number of launches, and resets the counters.  Used by bench.py for the roofline figure. */
int md2_profile_enable(md2_ctx* ctx, int32_t on);
int md2_profile_read(md2_ctx* ctx, float* total_ms, int64_t* launches);
/* md2_profile_enable(ctx, 2): time stamps around all three launches of the fused calls (prep | marching kernel | finish);
 * md2_profile_read_phases returns the three summed durations.  The event records between the launches add to the
 * gaps between them, so the three add up to a little more than an un-profiled step. */
int md2_profile_read_phases(md2_ctx* ctx, float* prep_ms, float* march_ms, float* finish_ms, int64_t* launches);

/* ---- A1  disparity_to_depth            src/utils.jl:175-179 ------------------------- */
int md2_disparity_to_depth_fwd(md2_ctx*, const float* disp, float* depth, int64_t count,
                               float min_depth, float max_depth, md2_stream);
int md2_disparity_to_depth_bwd(md2_ctx*, const float* disp, const float* gdepth, float* gdisp,
                               int64_t count, float min_depth, float max_depth, md2_stream);

/* ---- A2  Backproject(depth, invK)      src/utils.jl:41-65 ---------------------------
 * depth (1,P,N), invK (3,3) -> points (3,P,N) */
int md2_backproject_fwd(md2_ctx*, const float* depth, const float* invK, float* points,
                        int32_t W, int32_t H, int32_t N, md2_stream);
int md2_backproject_bwd(md2_ctx*, const float* gpoints, const float* invK, float* gdepth,
                        int32_t W, int32_t H, int32_t N, md2_stream);

/* ---- A3  Project(points, K, R, t)      src/utils.jl:67-99 ---------------------------
 * points (3,P,N), K (3,3), R (3,3,N), t (3,1,N) -> uv (2,P,N) normalised to (-1,1) */
int md2_project_fwd(md2_ctx*, const float* points, const float* K, const float* R, const float* t,
                    float* uv, int32_t W, int32_t H, int32_t N, md2_stream);
int md2_project_bwd(md2_ctx*, const float* points, const float* K, const float* R, const float* t,
                    const float* guv, float* gpoints, float* gR, float* gt,
                    int32_t W, int32_t H, int32_t N, md2_stream);

/* ---- A4/A5/A6  so3_exp_map, hat (+rrule), composeT   src/utils.jl:101-141,181-188 ---- */
int md2_so3_exp_map_fwd(md2_ctx*, const float* rvec, float* R, int32_t N, md2_stream);
int md2_so3_exp_map_bwd(md2_ctx*, const float* rvec, const float* gR, float* grvec, int32_t N, md2_stream);
int md2_hat_fwd(md2_ctx*, const float* rvec, float* S, int32_t N, md2_stream);
int md2_hat_bwd(md2_ctx*, const float* gS, float* grvec, int32_t N, md2_stream);
int md2_compose_T_fwd(md2_ctx*, const float* rvec, const float* tvec, int32_t invert,
                      float* R, float* t, int32_t N, md2_stream);
int md2_compose_T_bwd(md2_ctx*, const float* rvec, const float* tvec, int32_t invert,
                      const float* gR, const float* gt, float* grvec, float* gtvec, int32_t N, md2_stream);

/* ---- A16  NNlib.grid_sample (bilinear, align-corners)   call src/training.jl:56,
 *           test/runtests.jl:116.  padding_mode 0 = :zeros, 1 = :border.
 * input (W,H,C,N), grid (2,Wo,Ho,N) -> out (Wo,Ho,C,N).  ginput is ACCUMULATED. */
int md2_grid_sample_fwd(md2_ctx*, const float* input, const float* grid, float* out,
                        int32_t W, int32_t H, int32_t C, int32_t N, int32_t Wo, int32_t Ho,
                        int32_t padding_mode, md2_stream);
int md2_grid_sample_bwd(md2_ctx*, const float* input, const float* grid, const float* gout,
                        float* ginput, float* ggrid, int32_t W, int32_t H, int32_t C, int32_t N,
                        int32_t Wo, int32_t Ho, int32_t padding_mode, md2_stream);

/* ---- A17  NNlib.upsample_bilinear (align-corners)        call src/training.jl:45 ---- */
int md2_upsample_bilinear_fwd(md2_ctx*, const float* in, float* out, int32_t w, int32_t h,
                              int32_t W, int32_t H, int32_t CN, md2_stream);
int md2_upsample_bilinear_bwd(md2_ctx*, const float* gout, float* gin, int32_t w, int32_t h,
                              int32_t W, int32_t H, int32_t CN, md2_stream);

/* ---- A7  SSIM()(x, y)                  src/utils.jl:13-39 --------------------------- */
int md2_ssim_fwd(md2_ctx*, const float* x, const float* y, float* out,
                 int32_t W, int32_t H, int32_t C, int32_t N, md2_stream);
int md2_ssim_bwd(md2_ctx*, const float* x, const float* y, const float* gout, float* gx, float* gy,
                 int32_t W, int32_t H, int32_t C, int32_t N, md2_stream);

/* ---- A10-A13  photometric_loss / prediction_loss / automasking_loss / _apply_mask
 *               src/training.jl:1-19
 * out (W,H,1,N) = min( [mask,] photometric(pred_0,target), ..., photometric(pred_{S-1},target) ),
 * first index wins ties (findmin); argmin (optional, int32 (W,H,1,N)): -1 = mask, else s.
 * S = 1 and mask = NULL is photometric_loss itself.  pred pointers are (W,H,C,N) views with
 * an explicit per-image element stride, so frames of the 5-D input x (W,H,C,L,N) can be
 * passed without slicing (automasking_loss). */
int md2_photometric_min_fwd(md2_ctx*, int32_t S, const float* const* pred, const int64_t* pred_image_stride,
                            const float* target, int64_t target_image_stride, const float* mask,
                            float alpha, float* out, int32_t* argmin,
                            int32_t W, int32_t H, int32_t C, int32_t N, md2_stream);
/* gpred[s] (nullable, contiguous (W,H,C,N)), gtarget (nullable), gmask (nullable): overwritten */
int md2_photometric_min_bwd(md2_ctx*, int32_t S, const float* const* pred, const int64_t* pred_image_stride,
                            const float* target, int64_t target_image_stride, const float* mask,
                            float alpha, const float* gout, const int32_t* argmin /* from fwd */,
                            float* const* gpred, float* gtarget,
                            float* gmask, int32_t W, int32_t H, int32_t C, int32_t N, md2_stream);

/* ---- A8  smooth_loss(disparity, image) src/utils.jl:143-173 -------------------------
 * disparity (W,H,N), image (W,H,C,N) -> scalar (device).  normalize != 0 applies the
 * d / (mean_{W,H} d + 1e-7) of src/training.jl:64-65 first. */
int md2_smooth_loss_fwd(md2_ctx*, const float* disp, const float* image, int64_t image_stride,
                        float* out, int32_t normalize, int32_t W, int32_t H, int32_t C, int32_t N, md2_stream);
int md2_smooth_loss_bwd(md2_ctx*, const float* disp, const float* image, int64_t image_stride,
                        float gout, float* gdisp, float* gimage, int32_t normalize,
                        int32_t W, int32_t H, int32_t C, int32_t N, md2_stream);

/* ---- A14/A15  fused hot path ---------------------------------------------------------
 * warp (undefined in the reference; call src/simple_depth.jl:30-32, body inferred from
 * src/training.jl:48-57) and the train_loss tail (src/training.jl:29-77). */
typedef struct md2_vsl_desc {
    int32_t W, H, N, C, S, L;
    const float* target;  int64_t target_image_stride;        /* (W,H,C,N) view */
    const float* source[MD2_MAX_SOURCES];  int64_t source_image_stride[MD2_MAX_SOURCES];
    const float* disparity[MD2_MAX_SCALES];                   /* (w_i,h_i,1,N) */
    int32_t disp_w[MD2_MAX_SCALES], disp_h[MD2_MAX_SCALES];   /* upsampled to (W,H) if smaller */
    const float* K;  const float* invK;                       /* (3,3) device */
    int32_t pose_mode;       /* 0: rot = R (3,3,N), trans = t (3,1,N) as returned by composeT
                                1: rot = rvec (3,N), trans = tvec (3,1,N); composeT fused */
    const float* rot[MD2_MAX_SOURCES];
    const float* trans[MD2_MAX_SOURCES];
    int32_t invert[MD2_MAX_SOURCES];                          /* pose_mode 1: source_id < target_id */
    const float* automask;                                    /* (W,H,1,N) or NULL */
    float min_depth, max_depth;
    float smooth_weight[MD2_MAX_SCALES];    /* disparity_smoothness * scale_i */
    float loss_scale;                       /* 1 / L */
    int32_t normalize_disparity;            /* 1 in train_loss, 0 in slow_depth */
    /* outputs */
    float* loss;                                              /* device scalar */
    float* grad_disparity[MD2_MAX_SCALES];                    /* (w_i,h_i,1,N) */
    float* grad_rot[MD2_MAX_SOURCES];                         /* like rot */
    float* grad_trans[MD2_MAX_SOURCES];
    float* grad_source[MD2_MAX_SOURCES];    /* nullable; same view as source; ACCUMULATED */
    float* viz_warped[MD2_MAX_SOURCES];     /* nullable (W,H,C,N): warped sources, last scale */
    float* viz_loss;                        /* nullable (W,H,1,N): warp-loss map, last scale */
    float* saved;                           /* nullable (4,N,L): fwd -> bwd statistics */
    int32_t zero_grad_source;               /* != 0: the library zero-fills grad_source first (no caller memset) */
    /* Optional test hook (NULL in production; value + gradient calls with S = 2 only): the discrete decisions the
     * kernel took at every pixel of every scale, int32 (1+S, W, H, N, L) in Julia order, i.e. word k of pixel (x,y) of
     * image n at scale l is debug_choices[(((l*N + n)*H + y)*W + x)*(1+S) + k]:
     *   word 0: bits 0-1 selected source + 1 (0 = automask won); bit 2 + s*C + c: the SSIM clamp passed the gradient;
     *           bits 8 + 2*(s*C + c): sign of (warped - target) used by the L1 term (0: zero, 1: +, 2: -);
     *           bits 20-21 / 22-23: sign of d(x,y) - d(x+1,y) / d(x,y) - d(x,y+1) used by the smoothness term
     *   word 1+s: x0 | y0 << 14 | mask_x << 29 | mask_y << 30 of source s (0-based gather cell, clip-gradient masks)
     * A parity test evaluates the float64 oracle with exactly these decisions forced (tests/test_gpu_forced.py). */
    int32_t* debug_choices;
    /* != 0 and automask == NULL: the call forms the automask map itself from the un-warped source frames
     * (automasking_loss(ssim, x, target; source_ids), src/Monodepth.jl:159-164 / src/training.jl:9-11) as part of its launch
     * sequence -- the reference's separate pre-pass folded into the call.  The map is a constant of the loss, as in the
     * reference (it is computed outside `gradient`). */
    int32_t compute_automask;
    /* Camera intrinsics per image and their gradients (fields appended last: a zero-filled descriptor keeps one shared
     * camera and computes no intrinsics gradient).
     * per_image_K = 0: K / invK are one (3,3) pair for the batch; 1: K / invK are (3,3,N), element (i,j) of image n at
     * K[9n + 3j + i] (like R in pose_mode 0).
     * grad_K / grad_invK (nullable; OVERWRITTEN): dL/dK and dL/dinvK of the shape of K / invK -- (3,3) summed over sources
     * and images for a shared camera, (3,3,N) summed over sources per image.  invK is an independent input, as in the
     * reference (the call multiplies by the invK it is given; it never inverts K): dL/dK = sum G (R invK)^T + h t^T,
     * dL/dinvK = sum (K R)^T G over the (source, image) pairs, with R, t the pose actually used (after composeT).
     * Written by every call that writes grad_rot (value + gradient calls, the backward call, md2_warp_bwd); ignored by
     * the forward-only calls.  The sums are taken in a fixed (image, source) order in double precision, so both
     * gradients are bit-identical from run to run. */
    int32_t per_image_K;
    float* grad_K;
    float* grad_invK;
} md2_vsl_desc;

int md2_view_synthesis_loss_fwd(md2_ctx*, const md2_vsl_desc*, md2_stream);
int md2_view_synthesis_loss_bwd(md2_ctx*, const md2_vsl_desc*, float upstream, md2_stream);
/* value and gradient in one pass (gradient seeded with `seed`, normally 1) */
int md2_view_synthesis_loss_fwdbwd(md2_ctx*, const md2_vsl_desc*, float seed, md2_stream);

/* The same, for a caller whose buffers live in HOST memory (pinned for full speed): EVERY pointer of
 * the descriptor is a host pointer (inputs, K / invK, loss and all gradients; target / source /
 * grad_source keep their per-image strides).  This is the reference's per-step `x = device(x)` ...
 * `cpu(loss)` traffic (src/Monodepth.jl:156-176) folded into the call: the batch is cut into `groups`
 * groups of images whose host-to-device copies, kernels and device-to-host copies are pipelined over
 * three streams, and the pipeline is replayed as one CUDA graph while the descriptor stays the same.
 * Synchronous: returns when every output is in host memory.  saved / viz_* must be NULL. */
int md2_view_synthesis_loss_fwdbwd_host(md2_ctx*, const md2_vsl_desc* host_desc, float seed, int32_t groups);
/* Asynchronous form, for a caller that multi-buffers its batches (a data loader a step or two ahead): `submit` enqueues
 * the call on lane 0 .. MD2_HOST_LANES-1 and returns at once; `md2_host_wait(lane)` blocks until that call's outputs are in
 * host memory.  The lanes own separate streams, staging buffers, scratch and cached graphs, so the device-to-host copies
 * of step i overlap the host-to-device copies and kernels of step i+1 (submit(i+1, lane B) before wait(lane A)).
 * With one image group (groups = 1), inputs that lie in ONE stretch of host memory (frames, every disparity, automask
 * carved out of one pinned allocation) travel as a single copy.  So do the disparity gradients on the way back when the
 * L arrays lie back to back, with no gap between them; the call never writes a host byte outside its output arrays.  The host
 * buffers of a submitted descriptor must stay valid and untouched until its wait returns; submitting on a lane with an
 * uncollected call collects that call first.  md2_view_synthesis_loss_fwdbwd_host == submit + wait on lane 0. */
int md2_view_synthesis_loss_fwdbwd_host_submit(md2_ctx*, const md2_vsl_desc* host_desc, float seed, int32_t groups, int32_t lane);
int md2_host_wait(md2_ctx*, int32_t lane);

/* warp: disparity (W,H,1,N) -> S warped images (W,H,C,N); uses the desc fields
 * W,H,N,C,S, source*, disparity[0], K, invK, pose_*, rot, trans, invert, min/max_depth;
 * out[s] contiguous (W,H,C,N). */
int md2_warp_fwd(md2_ctx*, const md2_vsl_desc*, float* const* out, md2_stream);
/* gout[s] (W,H,C,N) -> grad_disparity[0], grad_rot, grad_trans, grad_source (accumulated), grad_K / grad_invK (nullable) */
int md2_warp_bwd(md2_ctx*, const md2_vsl_desc*, const float* const* gout, md2_stream);

/* ---- F1  Flux.Optimise.update!(ADAM, ...)   call src/Monodepth.jl:165-171, src/simple_depth.jl:20,43 --------------
 * One multi-tensor launch of the Flux ADAM rule (m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2;
 * p -= lr * m / (1 - b1^t) / (sqrt(v / (1 - b2^t)) + eps)) over n <= MD2_ADAM_MAX_TENSORS device tensors
 * (params[k], grads[k] with counts[k] elements; the arrays params / grads / counts themselves are HOST arrays).
 * grads are multiplied by grad_scale first (1 / world size after a SUM all-reduce).
 * Optimiser state is caller-owned device memory, which is what a checkpoint saves and restores:
 *   state  2 * sum(counts) floats: [m of the concatenated tensors | v of the concatenated tensors], zero-initialised
 *   clock  2 int64, zero-initialised: clock[0] = updates applied so far (t - 1; advanced on the device, so the call
 *          can be replayed from a CUDA graph), clock[1] = internal arrival counter (always 0 between launches) */
int md2_adam_step(md2_ctx*, int32_t n, float* const* params, const float* const* grads, const int64_t* counts,
                  float* state, int64_t* clock, float lr, float beta1, float beta2, float eps, float grad_scale, md2_stream);

/* ---- A15  slow_depth   src/simple_depth.jl:1-62 ---------------------------------------------------------------
 * The reference's single-triplet optimiser: `iters` iterations of { value + gradient of the objective described by
 * the descriptor; ADAM update of disparity[0] (W,H,1,N), rot[s] = rvec (3,N), trans[s] = tvec (3,1,N) IN PLACE }.
 * Descriptor: L = 1 with a full-resolution disparity, pose_mode = 1, loss / grad_disparity[0] / grad_rot / grad_trans
 * are scratch the call overwrites (the reference's objective is normalize_disparity = 0, smooth_weight[0] = 1,
 * loss_scale = 1: mean(prediction_loss) + smooth_loss).  state / clock as in md2_adam_step for the tensor order
 * disparity, rvec_0, tvec_0, rvec_1, tvec_1; loss_history (nullable, device, history_len floats) receives the
 * objective value of update number t at index t = clock[0] at that time (values beyond history_len are dropped).
 * One iteration is four launches captured once into a CUDA graph and replayed; the loop is ordered after the work
 * already enqueued on `stream` and before anything enqueued afterwards, and does not synchronise the host.
 * per_image_K is accepted (N = 1 here); grad_K / grad_invK must be NULL (the intrinsics are not among the optimised
 * tensors). */
int md2_slow_depth(md2_ctx*, const md2_vsl_desc*, int32_t iters, float lr, float beta1, float beta2, float eps,
                   float* state, int64_t* clock, float* loss_history, int64_t history_len, md2_stream);

#ifdef __cplusplus
}
#endif
#endif /* MD2_H */
