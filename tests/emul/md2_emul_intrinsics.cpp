// Test-only: the host emulation of md2_emul.cpp with a camera per image and the intrinsics gradients.  The orchestration
// of md2_emul.cpp is reused as it is; its two calls into the pose code are routed through the wrappers below, which give
// the pose inputs the descriptor's per-image K stride and, after each (source, image)'s pose finalisation, form that pair's
// contribution to dL/dK | dL/dinvK (intrinsics_part) -- what the finish kernel's pose blocks do.  The fixed-order
// reduction (reduce_intrinsics) then writes grad_K / grad_invK as the last pose block does on the device.
#include <vector>

#include "../../include/md2.h"
#include "../../monodepth2.jl_b200/csrc/md2_fused.cuh"

namespace md2 {
static int g_kstride = 0, g_N = 1;
static std::vector<double> g_kpart;   // (S*N, 18)

inline void prepare_pose_one_k(const PoseIO& io, int s, int n, float* ab, float* eb = nullptr) {
    PoseIO q = io;
    q.kstride = g_kstride;
    prepare_pose_one(q, s, n, ab, eb);
}
inline void finalize_pose_k(const PoseIO& io, int s, int n, const double* G, const double* h) {
    PoseIO q = io;
    q.kstride = g_kstride;
    finalize_pose(q, s, n, G, h);
    intrinsics_part(q, s, n, G, h, g_kpart.data() + ((size_t)s * g_N + n) * 18);
}
}  // namespace md2

#define prepare_pose_one prepare_pose_one_k
#define finalize_pose finalize_pose_k
#include "md2_emul.cpp"
#undef prepare_pose_one
#undef finalize_pose

// the march2 emulation (value + gradient) with desc->per_image_K, desc->grad_K / grad_invK honoured
extern "C" int md2_emul_march2_intrinsics(const md2_vsl_desc* d, int mode, float gloss, int R) {
    g_kstride = d->per_image_K ? 9 : 0;
    g_N = d->N;
    g_kpart.assign((size_t)18 * d->S * d->N, 0.0);
    const int rc = emul_vsl(d, mode, gloss, 2, R);
    if (rc == 0 && mode != 0) {
        IntrIO k{d->grad_K, d->grad_invK, g_kpart.data(), nullptr};
        reduce_intrinsics(k, g_kstride, d->S, d->N);
    }
    return rc;
}
