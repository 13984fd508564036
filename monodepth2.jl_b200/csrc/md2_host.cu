// Host-buffer entry point of the fused view-synthesis loss: md2_view_synthesis_loss_fwdbwd_host.
//
// The reference moves every batch to the device with `x = device(x)` and reads the loss back with
// `cpu(loss)` once per step (src/Monodepth.jl:156-176).  This entry point does the same for a caller
// whose buffers are in (pinned) host memory, without a per-step serial copy -> compute -> copy chain:
// the batch is cut into groups of images (the path is independent per image, DESIGN.md section 5) that
// are pipelined over three streams -- the host-to-device copies of group k+1 overlap the kernels of
// group k and the device-to-host copies of group k-1 -- and the whole pipeline (2-D strided copies,
// three kernels per group, events) is captured once per distinct descriptor into a CUDA graph, so a
// step is one cudaGraphLaunch + one synchronisation.
#include <string.h>

#include "md2_common.cuh"
#include "md2_fused.cuh"

namespace md2 {

int run_vsl(md2_ctx* ctx, const md2_vsl_desc* d, int mode, float gloss, cudaStream_t st);   // md2_fused.cu

constexpr int HOST_MAX_GROUPS = 16;

struct HostPath {
    cudaStream_t s_in = nullptr, s_run = nullptr, s_out = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_in0 = nullptr, ev_in[HOST_MAX_GROUPS] = {}, ev_done[HOST_MAX_GROUPS] = {},
                ev_join_in = nullptr, ev_join_run = nullptr;
    char* dbuf = nullptr;          // device staging of every input and output of one call
    size_t dbytes = 0;
    float* hsmall = nullptr;       // pinned staging of the small inputs (K, invK, poses) and outputs (pose gradients, partial losses)
    size_t hsmall_floats = 0;
    cudaGraphExec_t exec = nullptr;
    md2_vsl_desc key;              // descriptor the graph was captured for
    int key_groups = 0;
    float key_seed = 0.f;
    int64_t key_ws_gen = -1;       // ctx workspace generation the graph was captured with (the graph holds those pointers)
    bool have_key = false;
    // a submitted call whose outputs have not been collected yet (md2_host_wait)
    bool pending = false;
    md2_vsl_desc pend_desc;
    int pend_groups = 0;
    size_t pend_small_in = 0;
};

static HostPath* host_path(md2_ctx* ctx, int lane) {
    if (!ctx->host[lane]) {
        HostPath* h = new HostPath();
        bool ok = cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking) == cudaSuccess &&
                  cudaStreamCreateWithFlags(&h->s_run, cudaStreamNonBlocking) == cudaSuccess &&
                  cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking) == cudaSuccess &&
                  true;
        cudaEvent_t* evs[] = {&h->ev_fork, &h->ev_in0, &h->ev_join_in, &h->ev_join_run};
        for (cudaEvent_t* e : evs) ok = ok && cudaEventCreateWithFlags(e, cudaEventDisableTiming) == cudaSuccess;
        for (int k = 0; k < HOST_MAX_GROUPS; ++k)
            ok = ok && cudaEventCreateWithFlags(&h->ev_in[k], cudaEventDisableTiming) == cudaSuccess &&
                 cudaEventCreateWithFlags(&h->ev_done[k], cudaEventDisableTiming) == cudaSuccess;
        if (!ok) {
            set_error("host path: stream / event / pinned-memory creation failed: %s", cudaGetErrorString(cudaGetLastError()));
            delete h;
            return nullptr;
        }
        ctx->host[lane] = h;
    }
    return static_cast<HostPath*>(ctx->host[lane]);
}

static void host_lane_destroy(md2_ctx* ctx, int lane) {
    HostPath* h = static_cast<HostPath*>(ctx->host[lane]);
    if (!h) return;
    if (h->exec) cudaGraphExecDestroy(h->exec);
    if (h->dbuf) cudaFree(h->dbuf);
    if (h->hsmall) cudaFreeHost(h->hsmall);
    cudaStreamDestroy(h->s_in); cudaStreamDestroy(h->s_run); cudaStreamDestroy(h->s_out);
    cudaEvent_t evs[] = {h->ev_fork, h->ev_in0, h->ev_join_in, h->ev_join_run};
    for (cudaEvent_t e : evs) cudaEventDestroy(e);
    for (int k = 0; k < HOST_MAX_GROUPS; ++k) { cudaEventDestroy(h->ev_in[k]); cudaEventDestroy(h->ev_done[k]); }
    delete h;
    ctx->host[lane] = nullptr;
}

void host_path_destroy(md2_ctx* ctx) {
    for (int lane = 0; lane < MD2_HOST_LANES; ++lane) host_lane_destroy(ctx, lane);
}

// bump allocator over the staging buffer (256-byte aligned pieces)
struct Carver {
    char* base; size_t off = 0;
    float* take(size_t floats) {
        float* q = base ? reinterpret_cast<float*>(base + off) : nullptr;
        off += (floats * sizeof(float) + 255) & ~(size_t)255;
        return q;
    }
};

// device mirror of the host descriptor: frames, every scale, poses, outputs.  The small inputs (K, invK, poses) and
// the small outputs (pose gradients, one partial loss per group) are contiguous blocks that travel in one copy each
// through a pinned staging buffer; frames that are adjacent in host memory (the frames of one 5-D `x`) travel as
// one contiguous copy per image group and are addressed with strides on the device, like on the host.
struct Mirror {
    float *tgt, *src[MAX_S], *disp[MAX_L], *K, *invK, *rot[MAX_S], *trans[MAX_S], *automask;
    float *loss, *gdisp[MAX_L], *grot[MAX_S], *gtrans[MAX_S], *gsrc[MAX_S];
    float *gK, *giK;               // intrinsics gradients: (3,3,N) per image, or one (3,3) partial per image group
    float *small_in, *small_out;
    size_t small_in_floats, small_out_floats;
    bool xcontig;                  // frames travel as whole images of `xstride` floats starting at host pointer xbase
    const float* xbase; float* xall; int64_t xstride;
    int64_t xspan;                 // floats from xbase to the end of the last frame in use of one image
    // slab mode (one image group): every large input / every disparity gradient lies in ONE stretch of host memory
    // (a caller that carves its pinned buffers out of one allocation): the device mirror keeps the host layout and the
    // stretch travels as a single copy at the large-transfer rate of the link.  Inputs may leave small gaps between
    // arrays (read, never written); the disparity gradients must lie back to back
    bool in_slab, out_slab;
    const float* in_lo; float* in_dev; size_t in_floats;
    float* out_lo; float* out_dev; size_t out_floats;
};

// do the host ranges [p_k, p_k + n_k) tile one stretch of memory (gaps of at most `pad` floats)?  -> lowest address, span
static bool one_stretch(const float* const* p, const size_t* n, int cnt, size_t pad, const float** lo, size_t* span) {
    if (cnt < 2) return false;
    int order[2 + MAX_L];
    for (int i = 0; i < cnt; ++i) order[i] = i;
    for (int i = 1; i < cnt; ++i)
        for (int j = i; j > 0 && p[order[j]] < p[order[j - 1]]; --j) { const int t = order[j]; order[j] = order[j - 1]; order[j - 1] = t; }
    for (int i = 0; i + 1 < cnt; ++i) {
        const float* end = p[order[i]] + n[order[i]];
        if (p[order[i + 1]] < end || (size_t)(p[order[i + 1]] - end) > pad) return false;
    }
    *lo = p[order[0]];
    *span = (size_t)(p[order[cnt - 1]] + n[order[cnt - 1]] - p[order[0]]);
    return true;
}

static size_t carve(const md2_vsl_desc* d, char* base, Mirror& m, int groups) {
    Carver c{base};
    const size_t img = (size_t)d->C * d->W * d->H, N = d->N;
    const int pr = d->pose_mode == 0 ? 9 : 3;
    // frames: contiguous mode if target and sources are distinct frames of one block per image
    {
        const float* lo = d->target;
        const float* hi = d->target;
        bool same = true;
        for (int s = 0; s < d->S; ++s) {
            if (d->source[s] < lo) lo = d->source[s];
            if (d->source[s] > hi) hi = d->source[s];
            same = same && d->source_image_stride[s] == d->target_image_stride;
        }
        const int64_t st = d->target_image_stride;
        m.xcontig = same && st >= (int64_t)img && (hi - lo) + (int64_t)img <= st && st <= 4 * (int64_t)img * (d->S + 1);
        m.xbase = lo; m.xstride = st; m.xspan = (hi - lo) + (int64_t)img;
    }
    m.in_slab = m.out_slab = false;
    if (groups == 1 && m.xcontig) {
        const float* p[2 + MAX_L]; size_t n[2 + MAX_L]; int cnt = 0;
        p[cnt] = m.xbase; n[cnt++] = (size_t)(N - 1) * m.xstride + (size_t)m.xspan;
        for (int l = 0; l < d->L; ++l) { p[cnt] = d->disparity[l]; n[cnt++] = N * (size_t)d->disp_w[l] * d->disp_h[l]; }
        if (d->automask) { p[cnt] = d->automask; n[cnt++] = N * (size_t)d->W * d->H; }
        m.in_slab = one_stretch(p, n, cnt, 1024, &m.in_lo, &m.in_floats);
    }
    if (groups == 1 && d->L >= 2) {
        // outputs: only gradient arrays that lie back to back qualify.  The stretch is copied back whole, so any gap
        // between two arrays would be overwritten with the never-written device memory of its mirror.
        const float* p[MAX_L]; size_t n[MAX_L];
        bool all = true;
        for (int l = 0; l < d->L; ++l) { p[l] = d->grad_disparity[l]; n[l] = N * (size_t)d->disp_w[l] * d->disp_h[l]; all = all && p[l]; }
        const float* lo = nullptr;
        m.out_slab = all && one_stretch(p, n, d->L, 0, &lo, &m.out_floats);
        m.out_lo = const_cast<float*>(lo);
    }
    m.in_dev = m.in_slab ? c.take(m.in_floats) : nullptr;
    m.out_dev = m.out_slab ? c.take(m.out_floats) : nullptr;
    if (m.in_slab) {
        m.xall = m.in_dev ? m.in_dev + (m.xbase - m.in_lo) : nullptr;
        m.tgt = m.xall ? m.xall + (d->target - m.xbase) : nullptr;
        for (int s = 0; s < MAX_S; ++s) m.src[s] = (s < d->S && m.xall) ? m.xall + (d->source[s] - m.xbase) : nullptr;
    } else if (m.xcontig) {
        m.xall = c.take(N * (size_t)m.xstride);
        m.tgt = m.xall ? m.xall + (d->target - m.xbase) : nullptr;
        for (int s = 0; s < MAX_S; ++s) m.src[s] = (s < d->S && m.xall) ? m.xall + (d->source[s] - m.xbase) : nullptr;
    } else {
        m.xall = nullptr;
        m.tgt = c.take(N * img);
        for (int s = 0; s < MAX_S; ++s) m.src[s] = s < d->S ? c.take(N * img) : nullptr;
    }
    {   // grad_source mirrors use the device stride of the source frames (the kernels address both with one stride)
        bool any = false;
        for (int s = 0; s < d->S; ++s) any = any || d->grad_source[s] != nullptr;
        float* gall = (m.xcontig && any) ? c.take(N * (size_t)m.xstride) : nullptr;
        for (int s = 0; s < MAX_S; ++s) {
            const bool on = s < d->S && d->grad_source[s];
            if (m.xcontig) m.gsrc[s] = (on && gall) ? gall + (d->source[s] - m.xbase) : nullptr;   // (null in the sizing pass)
            else m.gsrc[s] = on ? c.take(N * img) : nullptr;
        }
    }
    for (int l = 0; l < MAX_L; ++l) {
        const bool on = l < d->L;
        const size_t px = on ? (size_t)d->disp_w[l] * d->disp_h[l] : 0;
        if (on && m.in_slab) m.disp[l] = m.in_dev ? m.in_dev + (d->disparity[l] - m.in_lo) : nullptr;
        else m.disp[l] = on ? c.take(N * px) : nullptr;
        if (on && m.out_slab) m.gdisp[l] = m.out_dev ? m.out_dev + (d->grad_disparity[l] - m.out_lo) : nullptr;
        else m.gdisp[l] = on ? c.take(N * px) : nullptr;
    }
    if (d->automask && m.in_slab) m.automask = m.in_dev ? m.in_dev + (d->automask - m.in_lo) : nullptr;
    else m.automask = d->automask ? c.take(N * (size_t)d->W * d->H) : nullptr;
    // small inputs: K, invK (9 floats each, 9 N per image), then per source rot, trans
    const size_t kf = d->per_image_K ? 9 * N : 9;
    m.small_in_floats = 2 * kf + (size_t)d->S * (pr + 3) * N;
    m.small_in = c.take(m.small_in_floats);
    m.K = m.small_in; m.invK = m.small_in ? m.small_in + kf : nullptr;
    // small outputs: per source grot, gtrans, the partial losses, then grad_K | grad_invK (per image, or one partial
    // per image group for a shared camera) when asked for
    const size_t gkf = (d->grad_K || d->grad_invK) ? (d->per_image_K ? 9 * N : 9 * (size_t)HOST_MAX_GROUPS) : 0;
    m.small_out_floats = (size_t)d->S * (pr + 3) * N + HOST_MAX_GROUPS + 2 * gkf;
    m.small_out = c.take(m.small_out_floats);
    for (int s = 0; s < MAX_S; ++s) {
        const bool on = s < d->S && m.small_in;
        m.rot[s] = on ? m.small_in + 2 * kf + (size_t)s * (pr + 3) * N : nullptr;
        m.trans[s] = on ? m.rot[s] + (size_t)pr * N : nullptr;
        m.grot[s] = on ? m.small_out + (size_t)s * (pr + 3) * N : nullptr;
        m.gtrans[s] = on ? m.grot[s] + (size_t)pr * N : nullptr;
    }
    m.loss = m.small_out ? m.small_out + (size_t)d->S * (pr + 3) * N : nullptr;
    m.gK = (m.loss && gkf) ? m.loss + HOST_MAX_GROUPS : nullptr;
    m.giK = m.gK ? m.gK + gkf : nullptr;
    return c.off;
}

// MD2_HOST_TRACE=1 (eager mode only): time stamps of the pipeline stages, printed to stderr
struct Trace {
    bool on = false;
    cudaEvent_t ev[128]; const char* what[128]; int idx[128]; int n = 0;
    void mark(cudaStream_t s, const char* w, int k) {
        if (!on || n >= 128) return;
        cudaEventCreate(&ev[n]); cudaEventRecord(ev[n], s); what[n] = w; idx[n] = k; ++n;
    }
    void dump() {
        if (!on) return;
        cudaDeviceSynchronize();
        for (int i = 1; i < n; ++i) { float ms = 0.f; cudaEventElapsedTime(&ms, ev[0], ev[i]); fprintf(stderr, "[md2 host trace] %-10s %2d  %8.1f us\n", what[i], idx[i], ms * 1e3f); }
        for (int i = 0; i < n; ++i) cudaEventDestroy(ev[i]);
        n = 0;
    }
};
static Trace g_trace;

#define MD2_H2D(dst, src, bytes) MD2_CHECK(cudaMemcpyAsync((dst), (src), (bytes), cudaMemcpyHostToDevice, h->s_in))
#define MD2_D2H(dst, src, bytes) MD2_CHECK(cudaMemcpyAsync((dst), (src), (bytes), cudaMemcpyDeviceToHost, h->s_out))

// enqueue the whole pipeline on the three streams (eagerly, or under stream capture)
static int enqueue(md2_ctx* ctx, HostPath* h, const md2_vsl_desc* d, const Mirror& m, float seed, int groups) {
    const int N = d->N, W = d->W, H = d->H, C = d->C, S = d->S, L = d->L;
    const size_t img = (size_t)C * W * H, imgb = img * sizeof(float);
    const int pr = d->pose_mode == 0 ? 9 : 3;
    // fork: the copy streams join the origin stream (s_run)
    g_trace.mark(h->s_run, "start", 0);
    MD2_CHECK(cudaEventRecord(h->ev_fork, h->s_run));
    MD2_CHECK(cudaStreamWaitEvent(h->s_in, h->ev_fork, 0));
    MD2_CHECK(cudaStreamWaitEvent(h->s_out, h->ev_fork, 0));
    // once per call: intrinsics and poses (one block, staged by run_host), the low-resolution disparities (small)
    MD2_H2D(m.small_in, h->hsmall, sizeof(float) * m.small_in_floats);
    if (m.in_slab) MD2_H2D(m.in_dev, m.in_lo, sizeof(float) * m.in_floats);     // frames, every disparity, automask: one copy
    for (int l = 0; l < L && !m.in_slab; ++l)
        if (d->disp_w[l] != W || d->disp_h[l] != H)
            MD2_H2D(m.disp[l], d->disparity[l], sizeof(float) * (size_t)N * d->disp_w[l] * d->disp_h[l]);
    g_trace.mark(h->s_in, "in-small", 0);
    MD2_CHECK(cudaEventRecord(h->ev_in0, h->s_in));
    MD2_CHECK(cudaStreamWaitEvent(h->s_run, h->ev_in0, 0));
    for (int k = 0; k < groups; ++k) {
        const int n0 = (int)((long long)N * k / groups), n1 = (int)((long long)N * (k + 1) / groups), nk = n1 - n0;
        // ---- inputs of group k: frames (strided host views -> dense), full-resolution disparities, automask
        if (m.in_slab) {
            // (everything travelled with the slab)
        } else if (m.xcontig) {
            // (not nk * xstride: xbase need not be the first frame of the per-image block, and the host buffer ends with
            // the last frame of the last image)
            MD2_H2D(m.xall + (size_t)n0 * m.xstride, m.xbase + (size_t)n0 * m.xstride,
                    sizeof(float) * ((size_t)(nk - 1) * m.xstride + (size_t)m.xspan));
        } else {
            MD2_CHECK(cudaMemcpy2DAsync(m.tgt + n0 * img, imgb, d->target + (size_t)n0 * d->target_image_stride,
                                        sizeof(float) * d->target_image_stride, imgb, nk, cudaMemcpyHostToDevice, h->s_in));
            for (int s = 0; s < S; ++s)
                MD2_CHECK(cudaMemcpy2DAsync(m.src[s] + n0 * img, imgb, d->source[s] + (size_t)n0 * d->source_image_stride[s],
                                            sizeof(float) * d->source_image_stride[s], imgb, nk, cudaMemcpyHostToDevice, h->s_in));
        }
        for (int l = 0; l < L && !m.in_slab; ++l)
            if (d->disp_w[l] == W && d->disp_h[l] == H)
                MD2_H2D(m.disp[l] + (size_t)n0 * W * H, d->disparity[l] + (size_t)n0 * W * H, sizeof(float) * (size_t)nk * W * H);
        if (d->automask && !m.in_slab) MD2_H2D(m.automask + (size_t)n0 * W * H, d->automask + (size_t)n0 * W * H, sizeof(float) * (size_t)nk * W * H);
        g_trace.mark(h->s_in, "in", k);
        MD2_CHECK(cudaEventRecord(h->ev_in[k], h->s_in));
        // ---- kernels of group k: the device descriptor of its images; loss_scale carries the group's share
        md2_vsl_desc g = *d;
        g.N = nk;
        const int64_t fst = m.xcontig ? m.xstride : (int64_t)img;   // per-image stride of the frames on the device
        g.target = m.tgt + n0 * fst; g.target_image_stride = fst;
        for (int s = 0; s < S; ++s) {
            g.source[s] = m.src[s] + n0 * fst; g.source_image_stride[s] = fst;
            g.rot[s] = m.rot[s] + (size_t)n0 * pr; g.trans[s] = m.trans[s] + (size_t)n0 * 3;
            g.grad_rot[s] = m.grot[s] + (size_t)n0 * pr; g.grad_trans[s] = m.gtrans[s] + (size_t)n0 * 3;
            g.grad_source[s] = m.gsrc[s] ? m.gsrc[s] + n0 * fst : nullptr;
            g.viz_warped[s] = nullptr;
        }
        for (int l = 0; l < L; ++l) {
            const size_t px = (size_t)d->disp_w[l] * d->disp_h[l];
            g.disparity[l] = m.disp[l] + n0 * px; g.grad_disparity[l] = m.gdisp[l] + n0 * px;
        }
        const size_t ko = d->per_image_K ? (size_t)9 * n0 : 0, go = d->per_image_K ? (size_t)9 * n0 : (size_t)9 * k;
        g.K = m.K + ko; g.invK = m.invK + ko;
        g.grad_K = d->grad_K ? m.gK + go : nullptr; g.grad_invK = d->grad_invK ? m.giK + go : nullptr;
        g.automask = m.automask ? m.automask + (size_t)n0 * W * H : nullptr;
        g.loss = m.loss + k; g.viz_loss = nullptr; g.saved = nullptr;
        g.loss_scale = d->loss_scale * (float)nk / (float)N;   // mean over the whole batch = sum of the group shares
        g.zero_grad_source = 1;
        MD2_CHECK(cudaStreamWaitEvent(h->s_run, h->ev_in[k], 0));
        g_trace.mark(h->s_run, "run-begin", k);
        if (run_vsl(ctx, &g, /*MODE_FWDBWD*/ 2, seed, h->s_run)) return 1;
        g_trace.mark(h->s_run, "run-end", k);
        MD2_CHECK(cudaEventRecord(h->ev_done[k], h->s_run));
        // ---- outputs of group k
        MD2_CHECK(cudaStreamWaitEvent(h->s_out, h->ev_done[k], 0));
        if (m.out_slab) MD2_D2H(m.out_lo, m.out_dev, sizeof(float) * m.out_floats);    // every disparity gradient: one copy
        for (int l = 0; l < L && !m.out_slab; ++l)
            if (d->disp_w[l] == W && d->disp_h[l] == H)
                MD2_D2H(d->grad_disparity[l] + (size_t)n0 * W * H, m.gdisp[l] + (size_t)n0 * W * H, sizeof(float) * (size_t)nk * W * H);
        for (int s = 0; s < S; ++s)
            if (m.gsrc[s])
                MD2_CHECK(cudaMemcpy2DAsync(d->grad_source[s] + (size_t)n0 * d->source_image_stride[s],
                                            sizeof(float) * d->source_image_stride[s], m.gsrc[s] + n0 * fst, sizeof(float) * fst, imgb, nk,
                                            cudaMemcpyDeviceToHost, h->s_out));
        g_trace.mark(h->s_out, "out", k);
    }
    // once per call: the small outputs of all groups
    for (int l = 0; l < L && !m.out_slab; ++l)
        if (d->disp_w[l] != W || d->disp_h[l] != H)
            MD2_D2H(d->grad_disparity[l], m.gdisp[l], sizeof(float) * (size_t)N * d->disp_w[l] * d->disp_h[l]);
    MD2_D2H(h->hsmall + m.small_in_floats, m.small_out, sizeof(float) * m.small_out_floats);   // pose gradients + partial losses
    g_trace.mark(h->s_out, "out-small", 0);
    // join: everything ends on the origin stream
    MD2_CHECK(cudaEventRecord(h->ev_join_in, h->s_in));
    MD2_CHECK(cudaEventRecord(h->ev_join_run, h->s_out));
    MD2_CHECK(cudaStreamWaitEvent(h->s_run, h->ev_join_in, 0));
    MD2_CHECK(cudaStreamWaitEvent(h->s_run, h->ev_join_run, 0));
    return 0;
}

// wait for the call in flight on a lane and move its small outputs (pose gradients, loss) into the caller's buffers
static int collect(md2_ctx* ctx, int lane) {
    HostPath* h = static_cast<HostPath*>(ctx->host[lane]);
    if (!h || !h->pending) return 0;
    MD2_CHECK(cudaStreamSynchronize(h->s_run));
    h->pending = false;
    const md2_vsl_desc* d = &h->pend_desc;
    const int pr = d->pose_mode == 0 ? 9 : 3;
    const float* q = h->hsmall + h->pend_small_in;
    for (int s = 0; s < d->S; ++s) {
        if (d->grad_rot[s]) memcpy(d->grad_rot[s], q, sizeof(float) * pr * d->N);
        q += (size_t)pr * d->N;
        if (d->grad_trans[s]) memcpy(d->grad_trans[s], q, sizeof(float) * 3 * d->N);
        q += (size_t)3 * d->N;
    }
    double loss = 0.0;
    for (int k = 0; k < h->pend_groups; ++k) loss += (double)q[k];
    *d->loss = (float)loss;
    q += HOST_MAX_GROUPS;
    if (d->grad_K || d->grad_invK) {   // per image: the rows as they are; shared: the group partials added in group order
        const size_t gkf = d->per_image_K ? (size_t)9 * d->N : (size_t)9 * HOST_MAX_GROUPS;
        float* outs[2] = {d->grad_K, d->grad_invK};
        for (int w = 0; w < 2; ++w, q += gkf) {
            if (!outs[w]) continue;
            if (d->per_image_K) { memcpy(outs[w], q, sizeof(float) * 9 * d->N); continue; }
            for (int e = 0; e < 9; ++e) {
                double a = 0.0;
                for (int k = 0; k < h->pend_groups; ++k) a += (double)q[9 * k + e];
                outs[w][e] = (float)a;
            }
        }
    }
    return 0;
}

// enqueue one call on a lane (its own streams, staging buffers, workspace bank and cached graph); returns at once
static int submit(md2_ctx* ctx, const md2_vsl_desc* d, float seed, int groups, int lane) {
    MD2_REQUIRE(d != nullptr, "null descriptor");
    MD2_REQUIRE(d->N >= 1 && d->S >= 1 && d->S <= MAX_S && d->L >= 1 && d->L <= MAX_L, "bad N / S / L");
    MD2_REQUIRE(d->target && d->K && d->invK && d->loss, "null target / K / invK / loss");
    MD2_REQUIRE(d->per_image_K == 0 || d->per_image_K == 1, "per_image_K must be 0 or 1");
    MD2_REQUIRE(!d->saved && !d->viz_loss && !d->viz_warped[0] && !d->viz_warped[1], "saved / viz outputs are not supported by the host entry point");
    MD2_REQUIRE(!d->debug_choices, "debug_choices is not supported by the host entry point");
    for (int s = 0; s < d->S; ++s) MD2_REQUIRE(d->source[s] && d->rot[s] && d->trans[s], "null source / pose");
    for (int l = 0; l < d->L; ++l) MD2_REQUIRE(d->disparity[l] && d->grad_disparity[l], "null disparity / grad_disparity");
    if (groups < 1) groups = 1;
    if (groups > HOST_MAX_GROUPS) groups = HOST_MAX_GROUPS;
    if (groups > d->N) groups = d->N;
    MD2_USE_DEVICE(ctx);
    MD2_REQUIRE(!ctx->prof_on, "kernel profiling (md2_profile_enable) is not available on the host entry point");
    HostPath* h = host_path(ctx, lane);
    if (!h) return 1;
    if (collect(ctx, lane)) return 1;          // a lane holds one call at a time: an uncollected one is finished first
    struct BankGuard { md2_ctx* c; int prev; ~BankGuard() { c->bank = prev; } } bank_guard{ctx, ctx->bank};
    ctx->bank = 1 + lane;
    Mirror m;
    const size_t need = carve(d, nullptr, m, groups);
    if (need > h->dbytes) {
        if (h->exec) { cudaGraphExecDestroy(h->exec); h->exec = nullptr; h->have_key = false; }
        if (h->dbuf) { MD2_CHECK(cudaDeviceSynchronize()); cudaFree(h->dbuf); h->dbuf = nullptr; h->dbytes = 0; }
        MD2_CHECK(cudaMalloc(&h->dbuf, need + need / 4));
        h->dbytes = need + need / 4;
    }
    carve(d, h->dbuf, m, groups);
    const int pr = d->pose_mode == 0 ? 9 : 3;
    if (m.small_in_floats + m.small_out_floats > h->hsmall_floats) {
        if (h->exec) { cudaGraphExecDestroy(h->exec); h->exec = nullptr; h->have_key = false; }
        if (h->hsmall) { MD2_CHECK(cudaDeviceSynchronize()); cudaFreeHost(h->hsmall); h->hsmall = nullptr; }
        h->hsmall_floats = 2 * (m.small_in_floats + m.small_out_floats);
        MD2_CHECK(cudaMallocHost(&h->hsmall, sizeof(float) * h->hsmall_floats));
    }
    {   // stage the small inputs: K, invK, per source rot, trans
        float* q = h->hsmall;
        const size_t kf = d->per_image_K ? (size_t)9 * d->N : 9;
        memcpy(q, d->K, kf * sizeof(float)); memcpy(q + kf, d->invK, kf * sizeof(float));
        q += 2 * kf;
        for (int s = 0; s < d->S; ++s) {
            memcpy(q, d->rot[s], sizeof(float) * pr * d->N); q += (size_t)pr * d->N;
            memcpy(q, d->trans[s], sizeof(float) * 3 * d->N); q += (size_t)3 * d->N;
        }
    }
    const bool same = h->have_key && h->exec && h->key_groups == groups && h->key_seed == seed && h->key_ws_gen == ctx->ws_gen[ctx->bank] &&
                      memcmp(&h->key, d, sizeof(*d)) == 0;
    if (!same) {
        if (h->exec) { cudaGraphExecDestroy(h->exec); h->exec = nullptr; }
        h->have_key = false;
        // first call for this descriptor: run eagerly (sizes every workspace, validates the arguments) ...
        g_trace.on = getenv("MD2_HOST_TRACE") != nullptr;
        if (enqueue(ctx, h, d, m, seed, groups)) return 1;
        if (g_trace.on) { MD2_CHECK(cudaStreamSynchronize(h->s_run)); g_trace.dump(); }
        g_trace.on = false;
        // ... then capture the same pipeline for the calls that follow.  (The capture is made now -- nothing executes
        // while capturing, it only needs the workspaces to have their final sizes, which the eager call ensured.)
        if (!getenv("MD2_HOST_NO_GRAPH")) {
            MD2_CHECK(cudaStreamSynchronize(h->s_run));
            cudaGraph_t graph = nullptr;
            const int64_t launches = ctx->launches;
            MD2_CHECK(cudaStreamBeginCapture(h->s_run, cudaStreamCaptureModeThreadLocal));
            const int rc = enqueue(ctx, h, d, m, seed, groups);
            const cudaError_t ce = cudaStreamEndCapture(h->s_run, &graph);
            ctx->launches = launches;   // nothing ran while capturing
            if (rc || ce != cudaSuccess || !graph) {
                if (graph) cudaGraphDestroy(graph);
                cudaGetLastError();
                if (rc) return 1;
                return set_error("host path: stream capture failed: %s", cudaGetErrorString(ce));
            }
            const cudaError_t ie = cudaGraphInstantiate(&h->exec, graph, 0);
            cudaGraphDestroy(graph);
            if (ie != cudaSuccess) { h->exec = nullptr; return set_error("host path: cudaGraphInstantiate failed: %s", cudaGetErrorString(ie)); }
            memcpy(&h->key, d, sizeof(*d)); h->key_groups = groups; h->key_seed = seed; h->have_key = true;   // (byte copy: the reuse test is a memcmp)
            h->key_ws_gen = ctx->ws_gen[ctx->bank];   // any later growth of the bank's workspaces invalidates the graph
        }
    } else {
        MD2_CHECK(cudaGraphLaunch(h->exec, h->s_run));
        ctx->launches += 3 * groups;
    }
    h->pending = true;
    memcpy(&h->pend_desc, d, sizeof(*d));
    h->pend_groups = groups;
    h->pend_small_in = m.small_in_floats;
    return 0;
}

}  // namespace md2

extern "C" {

int md2_view_synthesis_loss_fwdbwd_host(md2_ctx* ctx, const md2_vsl_desc* d, float seed, int32_t groups) {
    MD2_REQUIRE(ctx != nullptr, "null ctx");
    if (md2::submit(ctx, d, seed, groups, 0)) return 1;
    return md2::collect(ctx, 0);
}

int md2_view_synthesis_loss_fwdbwd_host_submit(md2_ctx* ctx, const md2_vsl_desc* d, float seed, int32_t groups, int32_t lane) {
    MD2_REQUIRE(ctx != nullptr, "null ctx");
    MD2_REQUIRE(lane >= 0 && lane < MD2_HOST_LANES, "lane must be in 0 .. MD2_HOST_LANES-1");
    return md2::submit(ctx, d, seed, groups, lane);
}

int md2_host_wait(md2_ctx* ctx, int32_t lane) {
    MD2_REQUIRE(ctx != nullptr, "null ctx");
    MD2_REQUIRE(lane >= 0 && lane < MD2_HOST_LANES, "lane must be in 0 .. MD2_HOST_LANES-1");
    MD2_USE_DEVICE(ctx);
    return md2::collect(ctx, lane);
}

}  // extern "C"
