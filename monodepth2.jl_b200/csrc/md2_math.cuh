// Per-pixel / per-pose maths of the view-synthesis loss path, shared by every kernel.
// All functions are __host__ __device__ so that tests/emul can run the very same code on
// the CPU (test infrastructure only; the product path is the CUDA build).
//
// Reference semantics restated here (file:line in pxl-th/Monodepth2.jl):
//   disparity_to_depth  src/utils.jl:175-179      Backproject  src/utils.jl:41-65
//   Project/normalize   src/utils.jl:67-99        so3_exp_map  src/utils.jl:101-117
//   hat + rrule         src/utils.jl:119-141      composeT     src/utils.jl:181-188
//   SSIM                src/utils.jl:13-39        grid_sample(:border)  call src/training.jl:56
#pragma once
#include <math.h>

#if defined(__CUDACC__)
#define MD2_HD __host__ __device__ __forceinline__
#else
#define MD2_HD inline
#endif

namespace md2 {

constexpr float SSIM_C1 = 1e-4f;  // 0.01^2  (src/utils.jl:20)
constexpr float SSIM_C2 = 9e-4f;  // 0.03^2
constexpr float PHOTO_ALPHA = 0.85f;  // src/training.jl:2
constexpr float PROJ_EPS = 1e-7f;  // src/utils.jl:97

// ---------------------------------------------------------------------------------------
// geometry: depth -> backproject -> rigid transform -> pinhole projection, pre-composed.
// cam = K (R (z K^-1 p) + t) = z (A p) + b  with A = K R K^-1, b = K t, p = (px, py, 1),
// px/py 1-based pixel centres.  u = cam_x / (cam_z + 1e-7), v likewise: 1-based pixel
// coordinates in the source frame.  The reference then normalises to (-1,1) and
// grid_sample un-normalises again (align-corners); the two cancel, so (u,v) feed the
// sampler directly.
// ---------------------------------------------------------------------------------------
struct Proj {
    float u, v;      // projected 1-based pixel coordinates
    float q;         // 1 / (cam_z + eps)
    float ap[3];     // A p  (= d cam / d z)
};

MD2_HD void project_ab(const float* __restrict__ ab /*12: A row-major, b*/, float px, float py,
                       float z, Proj& o) {
    o.ap[0] = fmaf(ab[0], px, fmaf(ab[1], py, ab[2]));
    o.ap[1] = fmaf(ab[3], px, fmaf(ab[4], py, ab[5]));
    o.ap[2] = fmaf(ab[6], px, fmaf(ab[7], py, ab[8]));
    const float c0 = fmaf(z, o.ap[0], ab[9]);
    const float c1 = fmaf(z, o.ap[1], ab[10]);
    const float c2 = fmaf(z, o.ap[2], ab[11]);
    o.q = 1.0f / (c2 + PROJ_EPS);
    o.u = c0 * o.q;
    o.v = c1 * o.q;
}

// adjoint of project_ab wrt cam given (du, dv):  cbar = (du q, dv q, -(du u + dv v) q)
MD2_HD void project_ab_bwd(const Proj& p, float du, float dv, float cbar[3]) {
    cbar[0] = du * p.q;
    cbar[1] = dv * p.q;
    cbar[2] = -(du * p.u + dv * p.v) * p.q;
}

// ---------------------------------------------------------------------------------------
// bilinear border-clamped sampling taps (NNlib.grid_sample padding_mode=:border,
// align-corners).  Input (u,v) 1-based; taps are 0-based indices.
// mask = 0 where the un-clipped coordinate is <= 1 or >= size (closed), as in the
// clip_coordinates gradient of the PyTorch kernel NNlib's was ported from.
// ---------------------------------------------------------------------------------------
struct Taps {
    int x0, x1, y0, y1;
    float fx, fy;   // fractional offsets in [0,1)
    float mx, my;   // clip-gradient masks
};

MD2_HD Taps border_taps(float u, float v, int W, int H) {
    Taps t;
    const float cu = fminf(fmaxf(u, 1.0f), (float)W) - 1.0f;  // 0-based, in [0, W-1]
    const float cv = fminf(fmaxf(v, 1.0f), (float)H) - 1.0f;
    t.mx = (u > 1.0f && u < (float)W) ? 1.0f : 0.0f;
    t.my = (v > 1.0f && v < (float)H) ? 1.0f : 0.0f;
    // the cell is kept inside the image (x0 <= W-2): at the last column the sample is expressed as
    // (x0 = W-2, fx = 1) instead of (x0 = W-1, fx = 0) -- same value, same image gradient, the
    // coordinate gradient is masked there anyway -- so that all four taps are always in range
    int x0 = (int)cu, y0 = (int)cv;                            // cu, cv >= 0: truncation == floor
    x0 = x0 < W - 2 ? x0 : W - 2;
    y0 = y0 < H - 2 ? y0 : H - 2;
    t.fx = cu - (float)x0;
    t.fy = cv - (float)y0;
    t.x0 = x0; t.y0 = y0; t.x1 = x0 + 1; t.y1 = y0 + 1;
    return t;
}

MD2_HD float bilerp(float v00, float v01, float v10, float v11, float fx, float fy) {
    const float top = fmaf(fx, v01 - v00, v00);
    const float bot = fmaf(fx, v11 - v10, v10);
    return fmaf(fy, bot - top, top);
}

// ---------------------------------------------------------------------------------------
// SSIM dissimilarity of one 3x3 window from CENTRED sums (x' = x - xc, y' = y - yc; the
// variances are shift invariant, which removes the E[x^2]-mu^2 cancellation of the
// reference's fp32 formula without changing the maths).
// x = predicted, y = target.  Returns clamp((1-S)/2, 0, 1).
// If coef != nullptr also returns (alpha, beta, gamma) with
//   dS/dx_j = alpha + beta x_j + gamma y_j  for a member pixel j (un-centred values)
// and *pass = 1 when the clamp passes the gradient (closed interval).
// ---------------------------------------------------------------------------------------
struct SsimWin {
    float s;                 // clamped dissimilarity
    float alpha, beta, gamma;
    float pass;
};

template <bool WITH_COEF>
MD2_HD SsimWin ssim_window(float xc, float yc, float sx, float sy, float sxx, float syy,
                           float sxy) {
    const float r9 = 1.0f / 9.0f;
    const float dx = sx * r9, dy = sy * r9;          // mu - centre
    const float mux = xc + dx, muy = yc + dy;
    const float vx = fmaf(-dx, dx, sxx * r9);
    const float vy = fmaf(-dy, dy, syy * r9);
    const float vxy = fmaf(-dx, dy, sxy * r9);
    // A and Cc (B and D) are formed so that identical inputs give bit-identical numerator and
    // denominator: ssim(x, x) is then exactly 0, as in the reference's own test.
    const float A = 2.0f * mux * muy + SSIM_C1;
    const float B = 2.0f * vxy + SSIM_C2;
    const float Cc = (mux * mux + muy * muy) + SSIM_C1;
    const float D = (vx + vy) + SSIM_C2;
    const float S = (A * B) / (Cc * D);
    const float raw = (1.0f - S) * 0.5f;
    SsimWin o;
    o.s = fminf(fmaxf(raw, 0.0f), 1.0f);
    if (WITH_COEF) {
        const float k = 2.0f / 9.0f;
        const float rC = 1.0f / Cc, rD = 1.0f / D;
        const float inv = rC * rD;
        o.pass = (raw >= 0.0f && raw <= 1.0f) ? 1.0f : 0.0f;
        o.beta = -k * S * rD;
        o.gamma = k * A * inv;
        o.alpha = k * (muy * (B - A) * inv - S * mux * rC + S * mux * rD);
    } else {
        o.pass = 0.f; o.alpha = o.beta = o.gamma = 0.f;
    }
    return o;
}

// align-corners bilinear resize taps (NNlib.upsample_bilinear, call src/training.jl:45):
// source coordinate = x * (w-1)/(W-1)
// The source coordinate is formed in exact integer arithmetic (x (w-1) = x0 (W-1) + rem, fx = rem / (W-1)): in float32 the
// product scale * x is only good to 3e-5 at x ~ 300, and that error of the interpolation weight moves the upsampled disparity
// -- and through it the sampling position of the warp -- by more than float32 rounding of the disparity itself.
MD2_HD void up_taps(int x, int w, int W, int& x0, int& x1, float& fx) {
    if (W <= 1) { x0 = 0; x1 = w > 1 ? 1 : 0; fx = 0.f; return; }
    const int den = W - 1, num = x * (w - 1);              // (< 2^31: W <= 12288, w <= W)
    int k = (int)((float)num * (1.0f / (float)den));       // within +-1 of the quotient
    int rem = num - k * den;
    if (rem < 0) { --k; rem += den; }
    if (rem >= den) { ++k; rem -= den; }
    x0 = k;
    fx = (float)rem / (float)den;
    if (x0 > w - 1) { x0 = w - 1; fx = 0.f; }
    x1 = x0 + 1 < w ? x0 + 1 : w - 1;
}
MD2_HD float up_scale(int w, int W) { return W > 1 ? (float)(w - 1) / (float)(W - 1) : 0.f; }

// reflect-pad(1) index map (src/utils.jl:26-27): -1 -> 1, n -> n-2
MD2_HD int reflect1(int i, int n) { return i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i); }

// ---------------------------------------------------------------------------------------
// poses (tiny, done in double): so3 exp, composeT, pre-composition and their adjoints.
// Matrices here are ROW-major 3x3 (m[3*i+j]).
// ---------------------------------------------------------------------------------------
MD2_HD void mat3_mul(const double* a, const double* b, double* c) {
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j)
            c[3 * i + j] = a[3 * i] * b[j] + a[3 * i + 1] * b[3 + j] + a[3 * i + 2] * b[6 + j];
}
MD2_HD void mat3_t(const double* a, double* c) {
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) c[3 * i + j] = a[3 * j + i];
}
MD2_HD void hat3(const double* r, double* k) {
    k[0] = 0;     k[1] = -r[2]; k[2] = r[1];
    k[3] = r[2];  k[4] = 0;     k[5] = -r[0];
    k[6] = -r[1]; k[7] = r[0];  k[8] = 0;
}

// f1 = sin(th)/max(th,1e-4), f2 = (1-cos(th))/max(th,1e-4)^2 and sin, cos, th themselves from th^2.
// For 1e-8 < th^2 < 1/4 (every realistic pose: the clamp is inactive there) the even power series
// are used -- no sqrt / sin / cos calls, whose double-precision slow paths dominated the serial
// pose blocks of the prep and finish kernels; otherwise the library functions.
MD2_HD void so3_factors(double t2, double& th, double& s, double& c, double& f1, double& f2) {
    if (t2 > 1e-8 && t2 < 0.25) {
        f1 = 1.0 + t2 * (-1.0 / 6 + t2 * (1.0 / 120 + t2 * (-1.0 / 5040 + t2 * (1.0 / 362880 + t2 * (-1.0 / 39916800 +
             t2 * (1.0 / 6227020800.0 + t2 * (-1.0 / 1307674368000.0 + t2 * (1.0 / 355687428096000.0))))))));
        f2 = 0.5 + t2 * (-1.0 / 24 + t2 * (1.0 / 720 + t2 * (-1.0 / 40320 + t2 * (1.0 / 3628800 + t2 * (-1.0 / 479001600 +
             t2 * (1.0 / 87178291200.0 + t2 * (-1.0 / 20922789888000.0 + t2 * (1.0 / 6402373705728000.0))))))));
        th = sqrt(t2);
        s = th * f1;
        c = 1.0 - t2 * f2;
    } else {
        th = sqrt(t2);
        const double ti = 1.0 / fmax(th, 1e-4);
        s = sin(th); c = cos(th);
        f1 = ti * s; f2 = ti * ti * (1.0 - c);
    }
}

// R = I + f1 K + f2 K^2, theta_inv = 1/max(theta, 1e-4)   (src/utils.jl:102-117)
MD2_HD void so3_exp(const double* r, double* R) {
    double K[9], K2[9];
    hat3(r, K);
    mat3_mul(K, K, K2);
    double th, s, c, f1, f2;
    so3_factors(r[0] * r[0] + r[1] * r[1] + r[2] * r[2], th, s, c, f1, f2);
    for (int i = 0; i < 9; ++i) R[i] = f1 * K[i] + f2 * K2[i] + ((i % 4 == 0) ? 1.0 : 0.0);
}

// adjoint of so3_exp: Rbar (row-major) -> rbar.  At theta == 0 the reference's sqrt gives a
// NaN gradient (README.md:47-49); here the theta-path contributes 0 there (documented
// deviation, DESIGN.md).
MD2_HD void so3_exp_bwd(const double* r, const double* Rb, double* rb) {
    double K[9], K2[9], Kt[9], T1[9], T2[9];
    hat3(r, K);
    mat3_mul(K, K, K2);
    mat3_t(K, Kt);
    double th, s, c, f1, f2;
    so3_factors(r[0] * r[0] + r[1] * r[1] + r[2] * r[2], th, s, c, f1, f2);
    const double tc = fmax(th, 1e-4);
    const double ti = 1.0 / tc;
    mat3_mul(Rb, Kt, T1);
    mat3_mul(Kt, Rb, T2);
    double Kb[9], f1b = 0, f2b = 0;
    for (int i = 0; i < 9; ++i) {
        Kb[i] = f1 * Rb[i] + f2 * (T1[i] + T2[i]);
        f1b += Rb[i] * K[i];
        f2b += Rb[i] * K2[i];
    }
    const double gate = th > 1e-4 ? 1.0 : 0.0;
    const double thb = f1b * (c * ti - gate * s * ti * ti) +
                       f2b * (s * ti * ti - gate * 2.0 * (1.0 - c) * ti * ti * ti);
    // hat pullback (src/utils.jl:130-141)
    rb[0] = Kb[7] - Kb[5];
    rb[1] = Kb[2] - Kb[6];
    rb[2] = Kb[3] - Kb[1];
    if (th > 0.0) {
        for (int i = 0; i < 3; ++i) rb[i] += thb * r[i] / th;
    }
}

// composeT(rvec, t, invert) -> (R_used, t_used)
MD2_HD void compose_T(const double* r, const double* t, int invert, double* R, double* tu) {
    double R0[9];
    so3_exp(r, R0);
    if (invert) {
        mat3_t(R0, R);
        for (int i = 0; i < 3; ++i) tu[i] = -(R[3 * i] * t[0] + R[3 * i + 1] * t[1] + R[3 * i + 2] * t[2]);
    } else {
        for (int i = 0; i < 9; ++i) R[i] = R0[i];
        for (int i = 0; i < 3; ++i) tu[i] = t[i];
    }
}

// adjoint of composeT: (Rbar_used, tbar_used) -> (rbar, tbar)
MD2_HD void compose_T_bwd(const double* r, const double* t, int invert, const double* Rub,
                          const double* tub, double* rb, double* tb) {
    double Rb[9];
    if (invert) {
        // R_used = R^T, t_used = -R_used t
        double R0[9];
        so3_exp(r, R0);
        double Rub2[9];
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) Rub2[3 * i + j] = Rub[3 * i + j] - tub[i] * t[j];
        mat3_t(Rub2, Rb);
        for (int i = 0; i < 3; ++i)
            tb[i] = -(R0[3 * i] * tub[0] + R0[3 * i + 1] * tub[1] + R0[3 * i + 2] * tub[2]);
    } else {
        for (int i = 0; i < 9; ++i) Rb[i] = Rub[i];
        for (int i = 0; i < 3; ++i) tb[i] = tub[i];
    }
    so3_exp_bwd(r, Rb, rb);
}

// A = K R K^-1, b = K t  (K, Kinv, R row-major doubles)
MD2_HD void precompose(const double* K, const double* Kinv, const double* R, const double* t,
                       float* ab) {
    double KR[9], A[9];
    mat3_mul(K, R, KR);
    mat3_mul(KR, Kinv, A);
    for (int i = 0; i < 9; ++i) ab[i] = (float)A[i];
    for (int i = 0; i < 3; ++i) ab[9 + i] = (float)(K[3 * i] * t[0] + K[3 * i + 1] * t[1] + K[3 * i + 2] * t[2]);
}

// The same, as a displacement: E = K R K^-1 - I (formed in double, so that the small entries of E keep their relative
// accuracy when rounded to float32) and b.  The hot kernel projects with cam = z (p + E p) + b and forms u - px directly:
// the projected coordinate is then accurate to float32 rounding of the DISPLACEMENT (a few pixels), not of the
// coordinate itself (hundreds of pixels: 3e-5 px at W = 416, 6e-5 at 1024 -- which shows up as 1e-4 .. 4e-3 relative
// errors of the pose gradients, sums of per-pixel terms with heavy cancellation).
MD2_HD void precompose_e(const double* K, const double* Kinv, const double* R, const double* t, float* eb) {
    // (K R Kinv - I with the caller's K and Kinv as they are -- not K (R - I) Kinv: the reference multiplies by the invK it
    // is given, and a float32 invK is the inverse of K only to 1e-7, which is 4e-5 px at the right-hand image border)
    double KR[9], A[9];
    mat3_mul(K, R, KR);
    mat3_mul(KR, Kinv, A);
    for (int i = 0; i < 9; ++i) eb[i] = (float)(A[i] - ((i % 4 == 0) ? 1.0 : 0.0));
    for (int i = 0; i < 3; ++i) eb[9 + i] = (float)(K[3 * i] * t[0] + K[3 * i + 1] * t[1] + K[3 * i + 2] * t[2]);
}

// adjoint of the pre-composition: G = sum cbar (z p)^T (3x3 row-major), h = sum cbar
//   Rbar_used = K^T G K^-T ,  tbar_used = K^T h
MD2_HD void precompose_bwd(const double* K, const double* Kinv, const double* G, const double* h,
                           double* Rub, double* tub) {
    double Kt[9], Kit[9], T[9];
    mat3_t(K, Kt);
    mat3_t(Kinv, Kit);
    mat3_mul(Kt, G, T);
    mat3_mul(T, Kit, Rub);
    for (int i = 0; i < 3; ++i) tub[i] = Kt[3 * i] * h[0] + Kt[3 * i + 1] * h[1] + Kt[3 * i + 2] * h[2];
}

// the same adjoint with respect to the intrinsics, K^-1 an independent input (R, t: the pose actually used)
//   Kbar = G (R K^-1)^T + h t^T ,  Kinvbar = (K R)^T G
MD2_HD void precompose_intr_bwd(const double* K, const double* Kinv, const double* R, const double* t, const double* G,
                                const double* h, double* Kb, double* Kib) {
    double RKi[9], RKit[9], KR[9], KRt[9];
    mat3_mul(R, Kinv, RKi);
    mat3_t(RKi, RKit);
    mat3_mul(G, RKit, Kb);
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) Kb[3 * i + j] += h[i] * t[j];
    mat3_mul(K, R, KR);
    mat3_t(KR, KRt);
    mat3_mul(KRt, G, Kib);
}

}  // namespace md2
