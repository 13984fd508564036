// Shared pieces of the fused view-synthesis loss (src/training.jl:42-70 and its Zygote pullback):
// the launch parameter block, per-pixel helpers, the smoothness / mean-disparity statistics, the
// loss assembly and the pose finalisation.  The hot kernel itself is md2_march.cuh.
// Everything here is __host__ __device__ so that tests/emul can run the same code on the CPU.
#pragma once
#include <stddef.h>
#include "md2_math.cuh"

namespace md2 {

constexpr int MAX_S = 2;   // source frames (reference: source_ids = [1,3])
constexpr int MAX_L = 8;   // decoder scales (reference: 4)
constexpr int NSTAT = 4;   // per (scale, image): warp sum, smooth-x sum, smooth-y sum, disparity sum

struct PoseIO {            // pose inputs / gradient outputs, Julia memory order
    int mode;              // 0: rot = R (3,3,N) col-major, trans = t ; 1: rot = rvec (3,N), trans = tvec
    int kstride;           // floats between the K / invK of consecutive images: 0 (one camera) or 9 (md2_vsl_desc.per_image_K)
    const float* rot[MAX_S];
    const float* trans[MAX_S];
    int invert[MAX_S];
    const float* K; const float* invK;   // (3,3[,N]) col-major
    float* grot[MAX_S];
    float* gtrans[MAX_S];
};
// (kstride sits in what was the padding after `mode`: the layout of FusedParams, which the marching kernels read, is unchanged)
static_assert(offsetof(PoseIO, rot) == 8 && sizeof(PoseIO) == 96, "PoseIO layout");

// intrinsics gradients (md2_vsl_desc.grad_K / grad_invK): every (source, image) leaves its 18 double contributions in
// `part`; the last to arrive (device arrival counter, reset by that last arrival) sums them in a fixed order
struct IntrIO {
    float* gK; float* giK;     // nullable outputs, the shape of K / invK
    double* part;              // (S*N, 18): Kbar | Kinvbar row-major of (source s, image n) at row s*N + n
    unsigned* count;           // arrival counter, 0 between launches
};

struct FusedParams {
    int W, H, N, L, S;
    // target frame (N,C,H,W) view: element (n,c,y,x) at tgt[n*tgt_ns + c*H*W + y*W + x]
    const float* tgt; long long tgt_ns;
    const float* src[MAX_S]; long long src_ns[MAX_S];
    float* gsrc[MAX_S];                 // nullable; same strides as src; accumulated (atomics)
    const float* disp[MAX_L];           // disparity (N,dh,dw) per scale at its NATIVE size
    int dw[MAX_L], dh[MAX_L];
    float* gdisp[MAX_L];                // (N,dh,dw): written (full-res) / accumulated (low-res, pre-zeroed)
    const float* automask;              // (N,H,W) or null   (src/training.jl:60-62)
    const float* pose_ab;               // (S,N,12) pre-composed A|b
    const float* pose_e;                // (S,N,12) the same as a displacement: E = A - I | b (precompose_e)
    const float* stats;                 // (L,N,NSTAT) forward sums, needed by the backward pass
    float* partial;                     // (L*N, segments, NPART) per-segment partial sums of the marching kernel
    float depth_a, depth_b;             // z = 1/(a d + b)   (src/utils.jl:175-179)
    float smooth_w[MAX_L];              // disparity_smoothness * scale_i  (src/training.jl:66-67)
    float loss_scale;                   // 1/L  (src/training.jl:77)
    float gloss;                        // upstream cotangent of the scalar loss
    int normalize_disp;                 // 1: d / (mean d + 1e-7) before smoothness (src/training.jl:64-65)
    float* viz_warped[MAX_S];           // optional (N,C,H,W) contiguous, last scale only
    float* viz_loss;                    // optional (N,H,W), last scale only
    // finalisation (finish kernel, md2_fused.cu)
    int mode;                           // 0 fwd, 1 bwd, 2 fwdbwd
    float* stats_out;                   // (L*N, NSTAT) written in modes 0 and 2
    float* saved;                       // nullable copy of stats_out for a later bwd
    float* loss;                        // nullable device scalar
    PoseIO pose;
    // marching-warp kernel (md2_march.cuh): rows per chunk, offset of this call's pose rows in the
    // constant-memory pose table, and every scale's disparity / gradient at FULL resolution (the
    // caller's buffer for a native-size scale, ctx scratch for a low-res decoder scale)
    int m_R, m_group, pose_slot;   // m_group: the short last chunks of a (scale, image) are cut into this many work items
    const float* dfull[MAX_L];
    float* gfull[MAX_L];
    // fused fwd+bwd call: per-block partial sums (Sx, Sy, sum d, -) of the prep kernel, (L, N, prep_nblk, 4);
    // null when the backward takes the statistics of an earlier forward from `stats`
    const float* prep_part;
    int prep_nblk;
    float usx[MAX_L], usy[MAX_L];       // up_scale(dw, W), up_scale(dh, H) of every scale (host-computed: no device divisions)
    // align-corners upsample taps of the low-resolution scales, tabulated once per shape on the host (up_taps is exact
    // integer arithmetic with a division per call): entry x of tap_x[l] / y of tap_y[l] = { i0, i1 (int bits), f, 0 }
    const float* tap_x[MAX_L]; const float* tap_y[MAX_L];
    // ... and their adjoint (gather form of the upsample's pullback): entry i of inv_x[l] / inv_y[l] = { lo, count, start
    // (int bits), 0 }: low-res index i receives full-res indices lo .. lo+count-1 with the weights inv_w[l][start ..]
    const float* inv_x[MAX_L]; const float* inv_y[MAX_L]; const float* inv_w[MAX_L];
    int* dbg;                           // optional test hook: the discrete decisions per pixel and scale (md2.h: debug_choices)
};

#if defined(__CUDA_ARCH__)
#define MD2_ATOMIC_ADD(p, v) atomicAdd((p), (v))
__device__ __forceinline__ float md2_rcp_approx(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
#define MD2_RCP_FAST(x) md2_rcp_approx(x)
#define MD2_EXP(x) __expf(x)
#else
#define MD2_ATOMIC_ADD(p, v) (*(p) += (v))
#define MD2_RCP_FAST(x) (1.0f / (x))
#define MD2_EXP(x) expf(x)
#endif

// reciprocal for the geometry (depth, perspective divide): approx + one Newton step, <= 1 ulp
MD2_HD float rcp_acc(float x) {
#if defined(__CUDA_ARCH__)
    const float r = md2_rcp_approx(x);
    return fmaf(r, fmaf(-x, r, 1.0f), r);
#else
    return 1.0f / x;
#endif
}

MD2_HD float sgnf(float v) { return (float)(v > 0.f) - (float)(v < 0.f); }

// disparity of scale `l` at full-resolution pixel (gx,gy): direct read or on-the-fly
// align-corners bilinear upsample (A17)
MD2_HD float disp_fullres(const float* __restrict__ dp, int dw, int dh, bool native, int W, int H_, int gx, int gy) {
    if (native) return dp[gy * W + gx];
    int x0, x1, y0, y1; float fx, fy;
    up_taps(gx, dw, W, x0, x1, fx);
    up_taps(gy, dh, H_, y0, y1, fy);
    return bilerp(dp[y0 * dw + x0], dp[y0 * dw + x1], dp[y1 * dw + x0], dp[y1 * dw + x1], fx, fy);
}

// geometry + sampler of one pixel for one source, used by the stand-alone `warp` operator (A15)
template <int C>
struct Sampler {
    struct Warped {
        float val[C], dix[C], diy[C];
    };
    static MD2_HD void project_pixel(const FusedParams& p, const float* ab, int gx, int gy, float z, Proj& pr, Taps& tp) {
        const float px = (float)(gx + 1), py = (float)(gy + 1);
        pr.ap[0] = fmaf(ab[0], px, fmaf(ab[1], py, ab[2]));
        pr.ap[1] = fmaf(ab[3], px, fmaf(ab[4], py, ab[5]));
        pr.ap[2] = fmaf(ab[6], px, fmaf(ab[7], py, ab[8]));
        const float c0 = fmaf(z, pr.ap[0], ab[9]);
        const float c1 = fmaf(z, pr.ap[1], ab[10]);
        const float c2 = fmaf(z, pr.ap[2], ab[11]);
        pr.q = rcp_acc(c2 + PROJ_EPS);
        pr.u = c0 * pr.q;
        pr.v = c1 * pr.q;
        tp = border_taps(pr.u, pr.v, p.W, p.H);
    }
    template <bool DERIV>
    static MD2_HD void gather(const FusedParams& p, int n, int s, const Taps& tp, Warped& w) {
        const long long HW = (long long)p.W * p.H;
        const float* base = p.src[s] + (long long)n * p.src_ns[s];
        const float* r0 = base + (tp.y0 * p.W + tp.x0);   // the 2x2 cell is always inside the image
        const float* r1 = r0 + p.W;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const float v00 = r0[c * HW], v01 = r0[c * HW + 1], v10 = r1[c * HW], v11 = r1[c * HW + 1];
            w.val[c] = bilerp(v00, v01, v10, v11, tp.fx, tp.fy);
            if (DERIV) {
                w.dix[c] = fmaf(tp.fy, (v11 - v10) - (v01 - v00), v01 - v00);
                w.diy[c] = fmaf(tp.fx, (v11 - v01) - (v10 - v00), v10 - v00);
            }
        }
    }
};

// adjoint of the align-corners bilinear upsample (A17) at low-res pixel (xi, yi): gather form,
// deterministic.  g is one full-resolution (H, W) gradient image.
MD2_HD float upsample_adjoint_at(const float* __restrict__ g, int w, int h, int W, int H, int xi, int yi) {
    const float sx = up_scale(w, W), sy = up_scale(h, H);
    int xlo = 0, xhi = W - 1, ylo = 0, yhi = H - 1;
    if (sx > 0.f) {
        xlo = (int)floorf((float)(xi - 1) / sx) - 1; xlo = xlo < 0 ? 0 : xlo;
        xhi = (int)ceilf((float)(xi + 1) / sx) + 1; xhi = xhi > W - 1 ? W - 1 : xhi;
    }
    if (sy > 0.f) {
        ylo = (int)floorf((float)(yi - 1) / sy) - 1; ylo = ylo < 0 ? 0 : ylo;
        yhi = (int)ceilf((float)(yi + 1) / sy) + 1; yhi = yhi > H - 1 ? H - 1 : yhi;
    }
    float acc = 0.f;
    for (int y = ylo; y <= yhi; ++y) {
        int y0, y1; float fy;
        up_taps(y, h, H, y0, y1, fy);
        const float wy = (y0 == yi ? 1.f - fy : 0.f) + (y1 == yi ? fy : 0.f);
        if (wy == 0.f) continue;
        float row = 0.f;
        for (int x = xlo; x <= xhi; ++x) {
            int x0, x1; float fx;
            up_taps(x, w, W, x0, x1, fx);
            const float wx = (x0 == xi ? 1.f - fx : 0.f) + (x1 == xi ? fx : 0.f);
            row = fmaf(wx, g[y * W + x], row);
        }
        acc = fmaf(wy, row, acc);
    }
    return acc;
}

// one full-resolution pixel's contribution to the smoothness sums and the disparity sum of
// every scale (src/utils.jl:159-173): the edge weights exp(-|dT|) are shared by all scales
template <int C>
MD2_HD void stats_pixel_all(const FusedParams& p, int n, int gx, int gy, float* v /*[L][3]: sx, sy, dsum*/) {
    const long long HW = (long long)p.W * p.H;
    const float* t = p.tgt + (long long)n * p.tgt_ns + gy * p.W + gx;
    const bool hx = gx + 1 < p.W, hy = gy + 1 < p.H;
    float wx = 0.f, wy = 0.f;
    if (hx) {
        float g = 0.f;
        for (int c = 0; c < C; ++c) g += fabsf(t[c * HW] - t[c * HW + 1]);
        wx = MD2_EXP(-g * (1.0f / C));
    }
    if (hy) {
        float g = 0.f;
        for (int c = 0; c < C; ++c) g += fabsf(t[c * HW] - t[c * HW + p.W]);
        wy = MD2_EXP(-g * (1.0f / C));
    }
    for (int l = 0; l < p.L; ++l) {
        const int dw = p.dw[l], dh = p.dh[l];
        const bool native = (dw == p.W && dh == p.H);
        const float* dp = p.disp[l] + (long long)n * dw * dh;
        const float usx = up_scale(dw, p.W), usy = up_scale(dh, p.H);
        const float d = disp_fullres(dp, dw, dh, native, p.W, p.H, gx, gy);
        v[3 * l + 2] += d;
        if (hx) v[3 * l + 0] += fabsf(d - disp_fullres(dp, dw, dh, native, p.W, p.H, gx + 1, gy)) * wx;
        if (hy) v[3 * l + 1] += fabsf(d - disp_fullres(dp, dw, dh, native, p.W, p.H, gx, gy + 1)) * wy;
    }
}

// one pixel's contribution to the smoothness sums and the disparity sum (stand-alone smooth_loss)
template <int C>
MD2_HD void stats_pixel(const float* d, const float* t, long long i, int W, int H, float& sx, float& sy, float& ds) {
    const long long HW = (long long)W * H;
    const int x = (int)(i % W), y = (int)(i / W);
    const float dc = d[i];
    ds += dc;
    if (x + 1 < W) {
        float g = 0.f;
        for (int c = 0; c < C; ++c) g += fabsf(t[c * HW + i] - t[c * HW + i + 1]);
        sx += fabsf(dc - d[i + 1]) * expf(-g * (1.0f / C));
    }
    if (y + 1 < H) {
        float g = 0.f;
        for (int c = 0; c < C; ++c) g += fabsf(t[c * HW + i] - t[c * HW + i + W]);
        sy += fabsf(dc - d[i + W]) * expf(-g * (1.0f / C));
    }
}

// loss = loss_scale * sum_i [ mean(warp_loss_i) + smooth_w_i * smooth_loss(dhat_i, target) ]
// from the per-(scale,image) sums {warp, Sx, Sy, dsum}   (src/training.jl:64-69,77)
MD2_HD float loss_from_stats(const float* stats, int W, int H, int N, int L, const float* smooth_w,
                             float loss_scale, int normalize_disp) {
    const double P = (double)W * H;
    const double cx = 1.0 / ((double)(W - 1) * H * N), cy = 1.0 / ((double)W * (H - 1) * N);
    double loss = 0.0;
    for (int i = 0; i < L; ++i) {
        double warp = 0.0, sm = 0.0;
        for (int n = 0; n < N; ++n) {
            const float* st = stats + ((long long)i * N + n) * NSTAT;
            warp += st[0];
            const double m = normalize_disp ? ((double)st[3] / P + 1e-7) : 1.0;
            sm += (cx * st[1] + cy * st[2]) / m;
        }
        loss += warp / (P * N) + (double)smooth_w[i] * sm;
    }
    return (float)(loss * loss_scale);
}

// K, invK of image n as row-major doubles
MD2_HD void load_K(const PoseIO& io, int n, double* K, double* Ki) {
    const float* Kn = io.K + io.kstride * n;     // (9 N < 2^31: N <= 65535)
    const float* Kin = io.invK + io.kstride * n;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) { K[3 * i + j] = (double)Kn[3 * j + i]; Ki[3 * i + j] = (double)Kin[3 * j + i]; }
}

// K, invK of image n and the pose (R, t) actually used for (source s, image n): composeT applied
MD2_HD void pose_used(const PoseIO& io, int s, int n, double* K, double* Ki, double* R, double* t) {
    load_K(io, n, K, Ki);
    if (io.mode == 0) {
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) R[3 * i + j] = (double)io.rot[s][9 * n + 3 * j + i];
        for (int k = 0; k < 3; ++k) t[k] = io.trans[s][3 * n + k];
    } else {
        double r[3], tv[3];
        for (int k = 0; k < 3; ++k) { r[k] = io.rot[s][3 * n + k]; tv[k] = io.trans[s][3 * n + k]; }
        compose_T(r, tv, io.invert[s], R, t);
    }
}

// pose gradients of one (source, image) from the accumulated G|h of all scales
MD2_HD void finalize_pose(const PoseIO& io, int s, int n, const double* G, const double* h) {
    double K[9], Ki[9];
    load_K(io, n, K, Ki);
    double Rub[9], tub[3];
    precompose_bwd(K, Ki, G, h, Rub, tub);
    if (io.mode == 0) {
        if (io.grot[s])
            for (int r = 0; r < 3; ++r)
                for (int c = 0; c < 3; ++c) io.grot[s][9 * n + 3 * c + r] = (float)Rub[3 * r + c];
        if (io.gtrans[s])
            for (int k = 0; k < 3; ++k) io.gtrans[s][3 * n + k] = (float)tub[k];
    } else {
        double r[3], tv[3], rb[3], tb[3];
        for (int k = 0; k < 3; ++k) { r[k] = io.rot[s][3 * n + k]; tv[k] = io.trans[s][3 * n + k]; }
        compose_T_bwd(r, tv, io.invert[s], Rub, tub, rb, tb);
        if (io.grot[s])
            for (int k = 0; k < 3; ++k) io.grot[s][3 * n + k] = (float)rb[k];
        if (io.gtrans[s])
            for (int k = 0; k < 3; ++k) io.gtrans[s][3 * n + k] = (float)tb[k];
    }
}

// the contributions of one (source, image) to the intrinsics gradients from the same G|h: Kbar | Kinvbar, 18 doubles
// row-major.  (Not inlined on the device: it runs once per (source, image) and would otherwise add to the register
// pressure of the kernels that call it.)
#if defined(__CUDACC__)
static __host__ __device__ __noinline__
#else
inline
#endif
void intrinsics_part(const PoseIO& io, int s, int n, const double* G, const double* h, double* kpart) {
    double K[9], Ki[9], R[9], t[3];
    pose_used(io, s, n, K, Ki, R, t);
    precompose_intr_bwd(K, Ki, R, t, G, h, kpart, kpart + 9);
}

// element e of grad_K | grad_invK (e < 18 * (kstride ? N : 1)) from the (S*N, 18) contributions: per image (summed over
// sources in source order) or, for a shared camera, over all pairs in (image, source) order; double sums, float outputs in
// Julia column-major order.  Every element is independent: a block forms them in parallel, one thread each.
MD2_HD void reduce_intrinsics_elem(const IntrIO& k, int kstride, int S, int N, int e) {
    const int m = e / 18, q = e - 18 * m;
    const int n0 = kstride ? m : 0, n1 = kstride ? m + 1 : N;
    double a = 0.0;
    for (int n = n0; n < n1; ++n)
        for (int s = 0; s < S; ++s) {
            const double* src = k.part + ((long long)s * N + n) * 18 + q;   // (written by other blocks of the launch)
#if defined(__CUDA_ARCH__)
            a += __ldcg(src);
#else
            a += *src;
#endif
        }
    const int r = q % 9, i = r / 3, j = r % 3;
    float* out = q < 9 ? k.gK : k.giK;
    if (out) out[9 * m + 3 * j + i] = (float)a;
}

MD2_HD void reduce_intrinsics(const IntrIO& k, int kstride, int S, int N) {
    for (int e = 0; e < 18 * (kstride ? N : 1); ++e) reduce_intrinsics_elem(k, kstride, S, N, e);
}

// [composeT] + pre-composition of one (source, image)
MD2_HD void prepare_pose_one(const PoseIO& io, int s, int n, float* ab, float* eb = nullptr) {
    double K[9], Ki[9], R[9], t[3];
    pose_used(io, s, n, K, Ki, R, t);
    precompose(K, Ki, R, t, ab);
    if (eb) precompose_e(K, Ki, R, t, eb);
}

}  // namespace md2
