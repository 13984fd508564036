/* Gradients of the view-synthesis loss with respect to the camera intrinsics K and invK, in the plain-C float64 style of
 * oracle/c_oracle.c (test infrastructure, NOT product code).  The file includes that oracle for its forward pieces
 * (projection, sampling, SSIM windows and their adjoint, forced decisions) and adds the reverse pass that reaches K and
 * invK, derived per pixel by the naive chain rule -- NOT from the kernels' pre-composed form (dL/dA = G, dL/db = h):
 *   cam = K Y, Y = R X + t, X = z invK p   =>   Kbar += cb Y^T ,  invKbar += z (R^T K^T cb) p^T
 * K and invK are independent inputs (the loss multiplies by the invK it is given).  One camera for the batch; a caller
 * with a camera per image evaluates image by image (the path is independent per image up to the 1/N of the means). */
#include "../oracle/c_oracle.c"

CO_API int co_vsl_intrinsics_grad(
    const double* x, int N, int L, int C, int H, int W,                 /* frames [N][L][C][H][W] */
    int n_scales, const double* const* disps, const int* dh, const int* dw, /* decoder outputs, each [N][1][dh][dw] */
    const double* rvecs, const double* tvecs,                            /* [S][N][3] */
    const double* K, const double* invK, int target_id, int S, const int* source_ids,
    double min_depth, double max_depth, const double* auto_loss,         /* [N][H][W] or NULL */
    double alpha, const int* choices,                                    /* NULL or [n_scales][N][H][W][1+S] */
    double* gK, double* ginvK)                                           /* [3][3] each, overwritten */
{
    if (H < 2 || W < 2 || S < 1 || n_scales < 1) return 1;
    const int HW = H * W, fs = 1 + S;
    dims_t g = {H, W, K, invK};
    const double up = 1.0 / n_scales;
    double* D = malloc(sizeof(double) * N * HW);
    double* warped = malloc(sizeof(double) * S * C * HW);
    double* pe = malloc(sizeof(double) * S * HW);
    int* sel = malloc(sizeof(int) * HW);
    cell_t* cells = malloc(sizeof(cell_t) * S * HW);
    double* wb = malloc(sizeof(double) * S * C * HW);
    double* gs = malloc(sizeof(double) * HW);
    double (*Ru)[3][3] = malloc(sizeof(double[3][3]) * S * N);
    double (*tu)[3] = malloc(sizeof(double[3]) * S * N);
    memset(gK, 0, sizeof(double) * 9);
    memset(ginvK, 0, sizeof(double) * 9);
    for (int s = 0; s < S; ++s)
        for (int n = 0; n < N; ++n)
            compose_T(rvecs + 3 * (s * N + n), tvecs + 3 * (s * N + n), source_ids[s] < target_id, Ru[s * N + n], tu[s * N + n]);
    for (int i = 0; i < n_scales; ++i) {
        if (dh[i] == H && dw[i] == W) memcpy(D, disps[i], sizeof(double) * N * HW);
        else co_upsample_bilinear(disps[i], N, dh[i], dw[i], H, W, D);
        for (int n = 0; n < N; ++n) {
            const double* tgt = x + ((long)(n * L + target_id) * C) * HW;
            const int* fc = choices ? choices + ((long)(i * N + n) * HW) * fs : NULL;
            /* forward: warp, photometric loss per source, selection (as co_view_synthesis_loss) */
            for (int s = 0; s < S; ++s) {
                const double* src = x + ((long)(n * L + source_ids[s]) * C) * HW;
                for (int p = 0; p < HW; ++p) {
                    double X[3], cam[3], gxn, gyn;
                    project_pixel(&g, Ru[s * N + n], tu[s * N + n], depth_of(D[n * HW + p], min_depth, max_depth), p % W + 1, p / W + 1,
                                  X, cam, &gxn, &gyn);
                    const cell_t c = fc ? cell_forced(gxn, gyn, H, W, fc[p * fs + 1 + s]) : cell_of(gxn, gyn, H, W);
                    cells[s * HW + p] = c;
                    for (int ch = 0; ch < C; ++ch) warped[(s * C + ch) * HW + p] = sample_plane(src + (long)ch * HW, H, W, c);
                }
                for (int p = 0; p < HW; ++p) {
                    double l1 = 0.0, ss = 0.0;
                    for (int ch = 0; ch < C; ++ch) {
                        const double* xw = warped + (s * C + ch) * HW;
                        l1 += fabs(tgt[ch * HW + p] - xw[p]);
                        ss += clamp01(ssim_raw(window(xw, tgt + (long)ch * HW, H, W, p / W, p % W)));
                    }
                    pe[s * HW + p] = alpha * (ss / C) + (1.0 - alpha) * (l1 / C);
                }
            }
            for (int p = 0; p < HW; ++p) {
                double v = pe[p];
                int k = 0;
                for (int s = 1; s < S; ++s)
                    if (pe[s * HW + p] < v) { v = pe[s * HW + p]; k = s; }
                if (auto_loss && auto_loss[n * HW + p] <= v) k = -1;
                sel[p] = fc ? (fc[p * fs] & 3) - 1 : k;
            }
            /* reverse: d loss / d warped (mean over (W, H, 1, N) of the selected loss, 1 / n_scales) */
            const double gpe = up / ((double)N * HW);
            memset(wb, 0, sizeof(double) * S * C * HW);
            for (int s = 0; s < S; ++s)
                for (int ch = 0; ch < C; ++ch) {
                    const double* xw = warped + (s * C + ch) * HW;
                    for (int p = 0; p < HW; ++p) {
                        const double gp = sel[p] == s ? gpe : 0.0;
                        gs[p] = gp * alpha / C;
                        const double sg = fc ? code_sign((fc[p * fs] >> (8 + 2 * (s * C + ch))) & 3) : sgn(xw[p] - tgt[ch * HW + p]);
                        wb[(s * C + ch) * HW + p] += gp * (1.0 - alpha) / C * sg;
                    }
                    ssim_plane_bwd(xw, tgt + (long)ch * HW, H, W, gs, wb + (s * C + ch) * HW, fc, fs, 2 + s * C + ch);
                }
            /* ... through the sampler to the pixel coordinates, the perspective divide, K and invK */
            for (int s = 0; s < S; ++s) {
                const double* src = x + ((long)(n * L + source_ids[s]) * C) * HW;
                const double (*R)[3] = Ru[s * N + n];
                const double* t = tu[s * N + n];
                for (int p = 0; p < HW; ++p) {
                    const cell_t c = cells[s * HW + p];
                    double ixb = 0.0, iyb = 0.0;
                    for (int ch = 0; ch < C; ++ch) {
                        const double gw = wb[(s * C + ch) * HW + p];
                        const double* im = src + (long)ch * HW;
                        const double v00 = tap_at(im, H, W, c.y0, c.x0), v01 = tap_at(im, H, W, c.y0, c.x0 + 1);
                        const double v10 = tap_at(im, H, W, c.y0 + 1, c.x0), v11 = tap_at(im, H, W, c.y0 + 1, c.x0 + 1);
                        ixb += gw * ((v01 - v00) * (1 - c.fy) + (v11 - v10) * c.fy);
                        iyb += gw * ((v10 - v00) * (1 - c.fx) + (v11 - v01) * c.fx);
                    }
                    const double ub = c.mx ? ixb * ((W - 1) * 0.5) * (2.0 / (W - 1.0)) : 0.0;   /* un-normalise, normalise */
                    const double vb = c.my ? iyb * ((H - 1) * 0.5) * (2.0 / (H - 1.0)) : 0.0;
                    if (ub == 0.0 && vb == 0.0) continue;
                    const double z = depth_of(D[n * HW + p], min_depth, max_depth);
                    double X[3], cam[3], gxn, gyn, Y[3], Yb[3], Xb[3];
                    const double pix[3] = {(double)(p % W + 1), (double)(p / W + 1), 1.0};
                    project_pixel(&g, R, t, z, p % W + 1, p / W + 1, X, cam, &gxn, &gyn);
                    const double q = 1.0 / (cam[2] + 1e-7);
                    const double cb[3] = {ub * q, vb * q, -(ub * cam[0] + vb * cam[1]) * q * q};
                    for (int a = 0; a < 3; ++a) Y[a] = R[a][0] * X[0] + R[a][1] * X[1] + R[a][2] * X[2] + t[a];
                    for (int a = 0; a < 3; ++a)
                        for (int b = 0; b < 3; ++b) gK[3 * a + b] += cb[a] * Y[b];                       /* cam = K Y */
                    for (int j = 0; j < 3; ++j) Yb[j] = K[j] * cb[0] + K[3 + j] * cb[1] + K[6 + j] * cb[2];
                    for (int b = 0; b < 3; ++b) Xb[b] = R[0][b] * Yb[0] + R[1][b] * Yb[1] + R[2][b] * Yb[2];
                    for (int a = 0; a < 3; ++a)
                        for (int b = 0; b < 3; ++b) ginvK[3 * a + b] += z * Xb[a] * pix[b];              /* X = z invK p */
                }
            }
        }
    }
    free(D); free(warped); free(pe); free(sel); free(cells); free(wb); free(gs); free(Ru); free(tu);
    return 0;
}
