# Monodepth2B200.jl -- Julia binding of libmd2_b200.so (include/md2.h) for pxl-th/Monodepth2.jl.
#
# The file is `include`d INSIDE `module Monodepth`, after the reference's own sources (INTEGRATION.md):
#
#     # src/Monodepth.jl, after  include("training.jl")
#     include(joinpath(ENV["MD2_B200_DIR"], "julia", "Monodepth2B200.jl"))   # submodule Monodepth.B200
#     using .B200: warp                      # the function src/simple_depth.jl:30 calls and the reference never defines
#
# It does NOT define functions of its own for the reference's entry points: it `import`s the reference's generic
# functions and callable structs from the enclosing module and ADDS METHODS to them that are more specific in the array
# type (`CuArray{Float32}`), plus `ChainRulesCore.rrule`s for those methods, exactly as the reference does for `hat`
# (src/utils.jl:130-141).  Dispatch then sends every Float32 GPU call of train() / slow_depth() to the CUDA kernels,
# while CPU arrays, Float64 arrays and the reference's tests (test/runtests.jl, which run on Array{Float64}) keep the
# reference's own methods.  Cotangents of vector / tuple arguments are returned as plain Vectors / Tuples.
#
# STATUS: written against include/md2.h and the reference's signatures and statically reviewed; NOT executed -- there is
# no Julia toolchain in the build image or on the GPU box.  The very same C ABI is exercised end to end from C
# (tests/cabi/harness.c) and from Python ctypes (monodepth2.jl_b200/_lib.py) by the -m gpu tests.
module B200

using CUDA
using ChainRulesCore
using Statistics: mean
import ChainRulesCore: rrule
# the reference's generics and types this file extends (src/utils.jl, src/training.jl, src/simple_depth.jl, src/Monodepth.jl)
import ..Monodepth: disparity_to_depth, so3_exp_map, hat, composeT, photometric_loss, prediction_loss, automasking_loss,
                    _apply_mask, smooth_loss, train_loss, slow_depth, save_disparity
import ..Monodepth: SSIM, Backproject, Project, TrainCache, Params, Pose

const LIB = get(ENV, "MD2_B200_LIB", joinpath(@__DIR__, "..", "csrc", "libmd2_b200.so"))
const CuF = CuArray{Float32}
const P32 = CuPtr{Float32}
const MAX_S, MAX_L = 2, 8

# ---------------------------------------------------------------------------------------------
# context / errors
# ---------------------------------------------------------------------------------------------
const CTX = Dict{Int, Ptr{Cvoid}}()

last_error() = unsafe_string(ccall((:md2_last_error, LIB), Cstring, ()))
check(status::Cint) = status == 0 ? nothing : error("md2: " * last_error())

function ctx()
    dev = CUDA.deviceid(CUDA.device())
    get!(CTX, dev) do
        h = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:md2_create, LIB), Cint, (Cint, Ptr{Ptr{Cvoid}}), dev, h))
        h[]
    end
end
stream() = Base.unsafe_convert(Ptr{Cvoid}, CUDA.stream().handle)
ptr(x::CuF) = pointer(x)
ptr(::Nothing) = P32(0)

# ---------------------------------------------------------------------------------------------
# A1 disparity_to_depth (src/utils.jl:175-179)
# ---------------------------------------------------------------------------------------------
function disparity_to_depth(disparity::CuF, min_depth, max_depth)
    out = similar(disparity)
    check(ccall((:md2_disparity_to_depth_fwd, LIB), Cint, (Ptr{Cvoid}, P32, P32, Int64, Cfloat, Cfloat, Ptr{Cvoid}),
                ctx(), disparity, out, length(disparity), min_depth, max_depth, stream()))
    out
end
function rrule(::typeof(disparity_to_depth), disparity::CuF, min_depth, max_depth)
    y = disparity_to_depth(disparity, min_depth, max_depth)
    function pb(Δ)
        g = similar(disparity)
        check(ccall((:md2_disparity_to_depth_bwd, LIB), Cint, (Ptr{Cvoid}, P32, P32, P32, Int64, Cfloat, Cfloat, Ptr{Cvoid}),
                    ctx(), disparity, CuF(unthunk(Δ)), g, length(disparity), min_depth, max_depth, stream()))
        NoTangent(), g, NoTangent(), NoTangent()
    end
    y, pb
end

# ---------------------------------------------------------------------------------------------
# A2 Backproject / A3 Project (src/utils.jl:41-99): methods on the REFERENCE's callable structs.  The reference stores
# no width / height: Backproject holds the (3, W*H) pixel grid, Project the (W-1, H-1) normaliser; both are read back
# once per object (cached by identity), never per call.
# ---------------------------------------------------------------------------------------------
const SIZE_CACHE = IdDict{Any, Tuple{Int, Int}}()
function image_size(b::Backproject)
    get!(SIZE_CACHE, b.coordinates) do
        last_px = Array(b.coordinates[:, end])                  # (W, H, 1): the grid is filled w = 1:W, h = 1:H (src/utils.jl:47-51)
        (round(Int, last_px[1]), round(Int, last_px[2]))
    end
end
function image_size(p::Project)
    get!(SIZE_CACHE, p.normalizer) do
        wh = vec(Array(p.normalizer))                           # (W - 1, H - 1), src/utils.jl:72
        (round(Int, wh[1]) + 1, round(Int, wh[2]) + 1)
    end
end
ChainRulesCore.@non_differentiable image_size(::Any)

function (b::Backproject)(depth::CuF, invK::CuF)            # depth (1,P,N), invK (3,3) -> (3,P,N)
    W, H = image_size(b)
    N = length(depth) ÷ (W * H)
    pts = CUDA.zeros(Float32, 3, W * H, N)
    check(ccall((:md2_backproject_fwd, LIB), Cint, (Ptr{Cvoid}, P32, P32, P32, Cint, Cint, Cint, Ptr{Cvoid}),
                ctx(), depth, invK, pts, W, H, N, stream()))
    pts
end
function rrule(b::Backproject, depth::CuF, invK::CuF)
    y = b(depth, invK)
    W, H = image_size(b)
    function pb(Δ)
        g = similar(depth)
        check(ccall((:md2_backproject_bwd, LIB), Cint, (Ptr{Cvoid}, P32, P32, P32, Cint, Cint, Cint, Ptr{Cvoid}),
                    ctx(), CuF(unthunk(Δ)), invK, g, W, H, size(y, 3), stream()))
        NoTangent(), g, NoTangent()
    end
    y, pb
end

function (p::Project)(points::CuF, K::CuF, R::CuF, t::CuF)  # (3,P,N),(3,3[,1]),(3,3,N),(3,1,N) -> (2,P,N)
    W, H = image_size(p)
    N = size(points, 3)
    uv = CUDA.zeros(Float32, 2, size(points, 2), N)
    check(ccall((:md2_project_fwd, LIB), Cint, (Ptr{Cvoid}, P32, P32, P32, P32, P32, Cint, Cint, Cint, Ptr{Cvoid}),
                ctx(), points, K, R, t, uv, W, H, N, stream()))
    uv
end
function rrule(p::Project, points::CuF, K::CuF, R::CuF, t::CuF)
    y = p(points, K, R, t)
    W, H = image_size(p)
    function pb(Δ)
        gp, gR, gt = similar(points), similar(R), similar(t)
        check(ccall((:md2_project_bwd, LIB), Cint,
                    (Ptr{Cvoid}, P32, P32, P32, P32, P32, P32, P32, P32, Cint, Cint, Cint, Ptr{Cvoid}),
                    ctx(), points, K, R, t, CuF(unthunk(Δ)), gp, gR, gt, W, H, size(points, 3), stream()))
        NoTangent(), gp, NoTangent(), gR, gt
    end
    y, pb
end

# ---------------------------------------------------------------------------------------------
# A4-A6 so3_exp_map / hat / composeT (src/utils.jl:101-141, 181-188)
# ---------------------------------------------------------------------------------------------
function so3_exp_map(rvec::CuF)
    N = size(rvec, 2); R = CUDA.zeros(Float32, 3, 3, N)
    check(ccall((:md2_so3_exp_map_fwd, LIB), Cint, (Ptr{Cvoid}, P32, P32, Cint, Ptr{Cvoid}), ctx(), rvec, R, N, stream()))
    R
end
function rrule(::typeof(so3_exp_map), rvec::CuF)
    R = so3_exp_map(rvec)
    function pb(Δ)
        g = similar(rvec)
        check(ccall((:md2_so3_exp_map_bwd, LIB), Cint, (Ptr{Cvoid}, P32, P32, P32, Cint, Ptr{Cvoid}),
                    ctx(), rvec, CuF(unthunk(Δ)), g, size(rvec, 2), stream()))
        NoTangent(), g
    end
    R, pb
end
function hat(rvec::CuF)
    N = size(rvec, 2); S = CUDA.zeros(Float32, 3, 3, N)
    check(ccall((:md2_hat_fwd, LIB), Cint, (Ptr{Cvoid}, P32, P32, Cint, Ptr{Cvoid}), ctx(), rvec, S, N, stream()))
    S
end
function rrule(::typeof(hat), v::CuF)                       # the reference's one hand-written rrule
    Y = hat(v)
    function hat_pullback(Δ)
        g = similar(v)
        check(ccall((:md2_hat_bwd, LIB), Cint, (Ptr{Cvoid}, P32, P32, Cint, Ptr{Cvoid}), ctx(), CuF(unthunk(Δ)), g, size(v, 2), stream()))
        NoTangent(), g
    end
    Y, hat_pullback
end
function composeT(rvec::CuF, t::CuF, invert::Bool)
    N = size(rvec, 2); R = CUDA.zeros(Float32, 3, 3, N); tu = similar(t)
    check(ccall((:md2_compose_T_fwd, LIB), Cint, (Ptr{Cvoid}, P32, P32, Cint, P32, P32, Cint, Ptr{Cvoid}),
                ctx(), rvec, t, invert, R, tu, N, stream()))
    R, tu
end
function rrule(::typeof(composeT), rvec::CuF, t::CuF, invert::Bool)
    y = composeT(rvec, t, invert)
    function pb(Δ)
        ΔR, Δt = unthunk(Δ)
        gR = ΔR isa AbstractZero ? P32(0) : ptr(CuF(ΔR)); gt = Δt isa AbstractZero ? P32(0) : ptr(CuF(Δt))
        gr, gtv = similar(rvec), similar(t)
        check(ccall((:md2_compose_T_bwd, LIB), Cint, (Ptr{Cvoid}, P32, P32, Cint, P32, P32, P32, P32, Cint, Ptr{Cvoid}),
                    ctx(), rvec, t, invert, gR, gt, gr, gtv, size(rvec, 2), stream()))
        NoTangent(), gr, gtv, NoTangent()
    end
    y, pb
end

# ---------------------------------------------------------------------------------------------
# A7 SSIM (src/utils.jl:13-39)
# ---------------------------------------------------------------------------------------------
function (ssim::SSIM)(x::CuF, y::CuF)                      # (more specific than the reference's (x::AbstractArray{T}, y::K))
    W, H, C, N = size(x); out = similar(x)
    check(ccall((:md2_ssim_fwd, LIB), Cint, (Ptr{Cvoid}, P32, P32, P32, Cint, Cint, Cint, Cint, Ptr{Cvoid}),
                ctx(), x, y, out, W, H, C, N, stream()))
    out
end
function rrule(ssim::SSIM, x::CuF, y::CuF)
    out = ssim(x, y)
    function pb(Δ)
        W, H, C, N = size(x); gx, gy = similar(x), similar(y)
        check(ccall((:md2_ssim_bwd, LIB), Cint, (Ptr{Cvoid}, P32, P32, P32, P32, P32, Cint, Cint, Cint, Cint, Ptr{Cvoid}),
                    ctx(), x, y, CuF(unthunk(Δ)), gx, gy, W, H, C, N, stream()))
        NoTangent(), gx, gy
    end
    out, pb
end

# ---------------------------------------------------------------------------------------------
# A10-A13 photometric_loss / prediction_loss / automasking_loss / _apply_mask (src/training.jl:1-19)
# ---------------------------------------------------------------------------------------------
function _photomin(preds::Vector{<:CuF}, strides::Vector{Int64}, target::CuF, tstride::Int64, α, dims)
    W, H, C, N = dims; S = length(preds)
    out = CUDA.zeros(Float32, W, H, 1, N); arg = CUDA.zeros(Int32, W, H, 1, N)
    pp = [ptr(p) for p in preds]
    check(ccall((:md2_photometric_min_fwd, LIB), Cint,
                (Ptr{Cvoid}, Cint, Ptr{P32}, Ptr{Int64}, P32, Int64, P32, Cfloat, P32, CuPtr{Int32}, Cint, Cint, Cint, Cint, Ptr{Cvoid}),
                ctx(), S, pp, strides, target, tstride, P32(0), α, out, arg, W, H, C, N, stream()))
    out, arg
end
function _photomin_rrule(preds::Vector{<:CuF}, target::CuF, α)
    W, H, C, N = size(target); chw = Int64(W * H * C); S = length(preds)
    out, arg = _photomin(preds, fill(chw, S), target, chw, α, size(target))
    function pb(Δ)
        gp = [similar(p) for p in preds]; gt = similar(target)
        check(ccall((:md2_photometric_min_bwd, LIB), Cint,
                    (Ptr{Cvoid}, Cint, Ptr{P32}, Ptr{Int64}, P32, Int64, P32, Cfloat, P32, CuPtr{Int32}, Ptr{P32}, P32, P32,
                     Cint, Cint, Cint, Cint, Ptr{Cvoid}),
                    ctx(), S, [ptr(p) for p in preds], fill(chw, S), target, chw, P32(0), α, CuF(unthunk(Δ)), arg,
                    [ptr(g) for g in gp], gt, P32(0), W, H, C, N, stream()))
        gp, gt
    end
    out, pb
end
photometric_loss(ssim, predicted::CuF, target::CuF; α = 0.85f0) =
    _photomin([predicted], [Int64(length(predicted) ÷ size(predicted, 4))], target, Int64(length(target) ÷ size(target, 4)), α, size(target))[1]
function rrule(::typeof(photometric_loss), ssim, predicted::CuF, target::CuF; α = 0.85f0)
    out, pb = _photomin_rrule([predicted], target, α)
    out, Δ -> ((gp, gt) = pb(Δ); (NoTangent(), NoTangent(), gp[1], gt))
end
prediction_loss(ssim, predictions, target::CuF) =
    _photomin(collect(predictions), fill(Int64(length(target) ÷ size(target, 4)), length(predictions)), target,
              Int64(length(target) ÷ size(target, 4)), 0.85f0, size(target))[1]
function rrule(::typeof(prediction_loss), ssim, predictions, target::CuF)
    out, pb = _photomin_rrule(collect(predictions), target, 0.85f0)
    out, Δ -> ((gp, gt) = pb(Δ); (NoTangent(), NoTangent(), predictions isa Tuple ? Tuple(gp) : gp, gt))   # plain Vector / Tuple cotangent
end
function automasking_loss(ssim, inputs::CuF, target::CuF; source_ids)      # inputs (W,H,C,L,N): frames passed as views
    W, H, C, L, N = size(inputs); fstride = W * H * C
    preds = [unsafe_wrap(CuArray, pointer(inputs, (i - 1) * fstride + 1), (W, H, C, 1)) for i in source_ids]
    _photomin(preds, fill(Int64(fstride * L), length(source_ids)), target, Int64(W * H * C), 0.85f0, (W, H, C, N))[1]
end
ChainRulesCore.@non_differentiable automasking_loss(::Any...)              # a constant in train() (src/Monodepth.jl:159-164)
# _apply_mask (src/training.jl:17-19) keeps the reference's method: `minimum(cat(mask, warp_loss; dims=3); dims=3)` runs on
# CuArrays as it is, and inside train_loss it is fused into the kernel anyway (mask first: it wins ties).

# ---------------------------------------------------------------------------------------------
# A8 smooth_loss (src/utils.jl:143-173)
# ---------------------------------------------------------------------------------------------
function _smooth(disparity::CuF, image::CuF, normalize::Bool)
    W, H, C, N = size(image); out = CUDA.zeros(Float32, 1)
    check(ccall((:md2_smooth_loss_fwd, LIB), Cint, (Ptr{Cvoid}, P32, P32, Int64, P32, Cint, Cint, Cint, Cint, Cint, Ptr{Cvoid}),
                ctx(), disparity, image, W * H * C, out, normalize, W, H, C, N, stream()))
    CUDA.@allowscalar out[1]
end
smooth_loss(disparity::CuF, image::CuF) = _smooth(disparity, image, false)        # disparity (W,H,N), image (W,H,C,N)
function rrule(::typeof(smooth_loss), disparity::CuF, image::CuF)
    y = _smooth(disparity, image, false)
    function pb(Δ)
        W, H, C, N = size(image); gd, gi = similar(disparity), similar(image)
        check(ccall((:md2_smooth_loss_bwd, LIB), Cint,
                    (Ptr{Cvoid}, P32, P32, Int64, Cfloat, P32, P32, Cint, Cint, Cint, Cint, Cint, Ptr{Cvoid}),
                    ctx(), disparity, image, W * H * C, Float32(unthunk(Δ)), gd, gi, false, W, H, C, N, stream()))
        NoTangent(), gd, gi
    end
    y, pb
end

# ---------------------------------------------------------------------------------------------
# A14 / A15 fused hot path: md2_vsl_desc mirror (include/md2.h), warp, view_synthesis_loss
# ---------------------------------------------------------------------------------------------
struct VslDesc
    W::Int32; H::Int32; N::Int32; C::Int32; S::Int32; L::Int32
    target::P32; target_image_stride::Int64
    source::NTuple{MAX_S, P32}; source_image_stride::NTuple{MAX_S, Int64}
    disparity::NTuple{MAX_L, P32}; disp_w::NTuple{MAX_L, Int32}; disp_h::NTuple{MAX_L, Int32}
    K::P32; invK::P32
    pose_mode::Int32
    rot::NTuple{MAX_S, P32}; trans::NTuple{MAX_S, P32}; invert::NTuple{MAX_S, Int32}
    automask::P32
    min_depth::Float32; max_depth::Float32
    smooth_weight::NTuple{MAX_L, Float32}; loss_scale::Float32; normalize_disparity::Int32
    loss::P32
    grad_disparity::NTuple{MAX_L, P32}
    grad_rot::NTuple{MAX_S, P32}; grad_trans::NTuple{MAX_S, P32}; grad_source::NTuple{MAX_S, P32}
    viz_warped::NTuple{MAX_S, P32}; viz_loss::P32
    saved::P32
    zero_grad_source::Int32
    debug_choices::CuPtr{Int32}          # test hook of the C ABI; always NULL here
    compute_automask::Int32              # != 0 with automask == NULL: the call forms the automask map itself
    per_image_K::Int32                   # 1: K / invK are (3,3,N), one camera per image
    grad_K::P32; grad_invK::P32          # nullable: dL/dK, dL/dinvK (the shape of K / invK; invK an independent input)
end
per_image(K) = ndims(K) == 3 && size(K, 3) > 1
pad(v, n, z) = ntuple(i -> i <= length(v) ? v[i] : z, n)
frameptr(x::CuF, id) = pointer(x, (id - 1) * size(x, 1) * size(x, 2) * size(x, 3) + 1)   # x (W,H,C,L,N), 1-based frame id

"""
    view_synthesis_loss(x, disparities, poses, K, invK; target_id, source_ids, scales, ...)

Everything of `train_loss` after `model(...)` (src/training.jl:29-77) in three kernel launches.
Returns `(loss::CuArray{Float32,1}, grads)` where `grads = (disparities, rvecs, tvecs, K, invK)` are the
gradients for a unit cotangent (the pullback scales them); the last two are `nothing` unless `grad_K`.
K / invK are (3,3) for one camera or (3,3,N) for one camera per image.
"""
function vsl_fwdbwd(x::CuF, disparities, rvecs, tvecs, K::CuF, invK::CuF; target_id, source_ids, scales,
                    min_depth, max_depth, disparity_smoothness, auto_loss = nothing, normalize = true,
                    smooth_weight = nothing, loss_scale = nothing, viz = false, compute_automask = false, grad_K = false)
    W, H, C, Lf, N = size(x); S = length(source_ids); L = length(disparities)
    loss = CUDA.zeros(Float32, 1)
    gd = [similar(d) for d in disparities]; gr = [similar(r) for r in rvecs]; gt = [similar(t) for t in tvecs]
    vw = viz ? [CUDA.zeros(Float32, W, H, C, N) for _ in 1:S] : CuF[]
    vl = viz ? CUDA.zeros(Float32, W, H, 1, N) : nothing
    gK = grad_K ? similar(K) : nothing; giK = grad_K ? similar(invK) : nothing
    sw = smooth_weight === nothing ? Float32[disparity_smoothness * s for s in scales[1:L]] : Float32.(smooth_weight)
    fs = Int64(W * H * C * Lf)
    desc = Ref(VslDesc(W, H, N, C, S, L, frameptr(x, target_id), fs,
        pad([frameptr(x, i) for i in source_ids], MAX_S, P32(0)), pad(fill(fs, S), MAX_S, Int64(0)),
        pad([ptr(d) for d in disparities], MAX_L, P32(0)), pad(Int32[size(d, 1) for d in disparities], MAX_L, Int32(0)),
        pad(Int32[size(d, 2) for d in disparities], MAX_L, Int32(0)), ptr(K), ptr(invK), Int32(1),
        pad([ptr(r) for r in rvecs], MAX_S, P32(0)), pad([ptr(t) for t in tvecs], MAX_S, P32(0)),
        pad(Int32[i < target_id for i in source_ids], MAX_S, Int32(0)), ptr(auto_loss),
        Float32(min_depth), Float32(max_depth), pad(sw, MAX_L, 0f0),
        Float32(loss_scale === nothing ? 1 / L : loss_scale), Int32(normalize), ptr(loss),
        pad([ptr(g) for g in gd], MAX_L, P32(0)), pad([ptr(g) for g in gr], MAX_S, P32(0)),
        pad([ptr(g) for g in gt], MAX_S, P32(0)), pad(P32[], MAX_S, P32(0)),
        pad([ptr(v) for v in vw], MAX_S, P32(0)), ptr(vl), P32(0), Int32(0), CuPtr{Int32}(0), Int32(compute_automask && auto_loss === nothing),
        Int32(per_image(K)), ptr(gK), ptr(giK)))
    GC.@preserve x disparities rvecs tvecs K invK auto_loss loss gd gr gt vw vl gK giK begin
        check(ccall((:md2_view_synthesis_loss_fwdbwd, LIB), Cint, (Ptr{Cvoid}, Ptr{VslDesc}, Cfloat, Ptr{Cvoid}),
                    ctx(), desc, 1f0, stream()))
    end
    loss, (gd, gr, gt, gK, giK), vw, vl
end

"""
    vsl_fwdbwd_host!(loss, grads, x, disparities, rvecs, tvecs, K, invK; groups = 2, kw...)

The same for a batch that lives in (pinned) HOST memory -- `Array{Float32}`s registered with `CUDA.Mem.pin` --: the
reference's per-step `x = device(x)` ... `cpu(loss)` (src/Monodepth.jl:156-176) folded into one synchronous call of
`md2_view_synthesis_loss_fwdbwd_host`, which pipelines image groups over copy / compute streams and replays the
pipeline as a CUDA graph while the arrays stay the same.  `loss::Vector{Float32}` (length 1) and `grads = (gd, gr, gt)`
are host arrays written in place.
"""
function vsl_fwdbwd_host!(loss::Vector{Float32}, grads, x::Array{Float32,5}, disparities, rvecs, tvecs,
                          K::Array{Float32}, invK::Array{Float32}; target_id, source_ids, scales, min_depth, max_depth,
                          disparity_smoothness, normalize = true, groups = 2, lane = nothing)
    W, H, C, Lf, N = size(x); S = length(source_ids); L = length(disparities)
    gd, gr, gt = grads
    hp(a) = a === nothing ? P32(0) : reinterpret(P32, pointer(a))
    fp(id) = reinterpret(P32, pointer(x, (id - 1) * W * H * C + 1))
    fs = Int64(W * H * C * Lf)
    desc = Ref(VslDesc(W, H, N, C, S, L, fp(target_id), fs,
        pad([fp(i) for i in source_ids], MAX_S, P32(0)), pad(fill(fs, S), MAX_S, Int64(0)),
        pad([hp(d) for d in disparities], MAX_L, P32(0)), pad(Int32[size(d, 1) for d in disparities], MAX_L, Int32(0)),
        pad(Int32[size(d, 2) for d in disparities], MAX_L, Int32(0)), hp(K), hp(invK), Int32(1),
        pad([hp(r) for r in rvecs], MAX_S, P32(0)), pad([hp(t) for t in tvecs], MAX_S, P32(0)),
        pad(Int32[i < target_id for i in source_ids], MAX_S, Int32(0)), P32(0),
        Float32(min_depth), Float32(max_depth), pad(Float32[disparity_smoothness * s for s in scales[1:L]], MAX_L, 0f0),
        Float32(1 / L), Int32(normalize), hp(loss),
        pad([hp(g) for g in gd], MAX_L, P32(0)), pad([hp(g) for g in gr], MAX_S, P32(0)),
        pad([hp(g) for g in gt], MAX_S, P32(0)), pad(P32[], MAX_S, P32(0)),
        pad(P32[], MAX_S, P32(0)), P32(0), P32(0), Int32(1), CuPtr{Int32}(0), Int32(0), Int32(per_image(K)), P32(0), P32(0)))
    GC.@preserve x disparities rvecs tvecs K invK loss gd gr gt begin
        if lane === nothing          # synchronous: returns when every output is in host memory
            check(ccall((:md2_view_synthesis_loss_fwdbwd_host, LIB), Cint, (Ptr{Cvoid}, Ptr{VslDesc}, Cfloat, Cint),
                        ctx(), desc, 1f0, Cint(groups)))
        else                         # asynchronous: enqueue on lane 0 .. 2 and return; collect with vsl_host_wait(lane).
            # The caller keeps every array of this call alive and untouched until then (a data loader one or two steps ahead)
            check(ccall((:md2_view_synthesis_loss_fwdbwd_host_submit, LIB), Cint, (Ptr{Cvoid}, Ptr{VslDesc}, Cfloat, Cint, Cint),
                        ctx(), desc, 1f0, Cint(groups), Cint(lane)))
            return nothing
        end
    end
    loss[1]
end
"""`vsl_host_wait(lane)`: block until the call submitted on `lane` has written its loss and gradients to the host arrays."""
vsl_host_wait(lane::Integer) = check(ccall((:md2_host_wait, LIB), Cint, (Ptr{Cvoid}, Cint), ctx(), Cint(lane)))

# the tail of train_loss as one differentiable function of (disparities, rvecs, tvecs)
function view_synthesis_loss(x, disparities, rvecs, tvecs, K, invK; kw...)
    loss, _, _, _ = vsl_fwdbwd(x, disparities, rvecs, tvecs, K, invK; kw...)
    CUDA.@allowscalar loss[1]
end
function rrule(::typeof(view_synthesis_loss), x, disparities, rvecs, tvecs, K, invK; kw...)
    loss, (gd, gr, gt, gK, giK), _, _ = vsl_fwdbwd(x, disparities, rvecs, tvecs, K, invK; kw..., grad_K = true)
    function pb(Δ)
        s = Float32(unthunk(Δ))
        # cotangents of Vector-of-array arguments are plain Vectors of arrays (what Zygote accumulates into);
        # K and invK get theirs too (learned intrinsics), invK as an input of its own as in the reference
        NoTangent(), NoTangent(), [s .* g for g in gd], [s .* g for g in gr], [s .* g for g in gt], s .* gK, s .* giK
    end
    (CUDA.@allowscalar loss[1]), pb
end

"""
`train_loss` (src/training.jl:21-78) for a Float32 batch on the GPU: a METHOD of the reference's own generic (more
specific in `x` than its `x::AbstractArray{T}`), taking the reference's `TrainCache` / `Params`; frame ids are 1-based.
`model(...)` is differentiated by Zygote as before; everything after it is one rrule.
"""
function train_loss(model, x::CuArray{Float32, 5}, auto_loss, cache::TrainCache, parameters::Params, do_visualization)
    disparities, poses = model(x, cache.source_ids, cache.target_id)
    kw = (; target_id = cache.target_id, source_ids = cache.source_ids, scales = cache.scales,
          min_depth = parameters.min_depth, max_depth = parameters.max_depth,
          disparity_smoothness = parameters.disparity_smoothness,
          auto_loss = parameters.automasking ? auto_loss : nothing,
          compute_automask = parameters.automasking && auto_loss === nothing)   # no map handed in: the call forms it itself
    rvecs = [p.rvec for p in poses]; tvecs = [p.tvec for p in poses]
    loss = view_synthesis_loss(x, collect(disparities), rvecs, tvecs, cache.K, cache.invK; kw...)
    if do_visualization     # forward-only second pass for the logging outputs (every 50 iterations)
        _, _, vw, vl = ChainRulesCore.ignore_derivatives() do
            vsl_fwdbwd(x, collect(disparities), rvecs, tvecs, cache.K, cache.invK; kw..., viz = true)
        end
        return loss, Array(disparities[end]), Array.(vw), Array(vl)
    end
    loss, nothing, nothing, nothing
end

"""
`warp` -- called at src/simple_depth.jl:30-32 but never defined by the reference; body as in
src/training.jl:48-57.  `Ps` = vector of `(R, t)` from `composeT`.  Returns the warped images.
"""
function warp(disp::CuF, x::CuF, Ps, backprojections, projections, invKs::CuF, Ks::CuF; min_depth, max_depth, source_ids)
    W, H, C, Lf, N = size(x); S = length(source_ids); fs = Int64(W * H * C * Lf)
    outs = [CUDA.zeros(Float32, W, H, C, N) for _ in 1:S]
    desc = Ref(_warp_desc(disp, x, Ps, invKs, Ks, min_depth, max_depth, source_ids, nothing))
    GC.@preserve disp x Ps invKs Ks outs begin
        check(ccall((:md2_warp_fwd, LIB), Cint, (Ptr{Cvoid}, Ptr{VslDesc}, Ptr{P32}, Ptr{Cvoid}), ctx(), desc, [ptr(o) for o in outs], stream()))
    end
    outs
end
function _warp_desc(disp, x, Ps, invKs, Ks, min_depth, max_depth, source_ids, grads)
    W, H, C, Lf, N = size(x); S = length(source_ids); fs = Int64(W * H * C * Lf); z = P32(0)
    gd, gR, gt = grads === nothing ? (z, fill(z, S), fill(z, S)) : (ptr(grads[1]), ptr.(grads[2]), ptr.(grads[3]))
    VslDesc(W, H, N, C, S, 1, z, 0, pad([frameptr(x, i) for i in source_ids], MAX_S, z), pad(fill(fs, S), MAX_S, Int64(0)),
            pad([ptr(disp)], MAX_L, z), pad(Int32[W], MAX_L, Int32(0)), pad(Int32[H], MAX_L, Int32(0)), ptr(Ks), ptr(invKs),
            Int32(0), pad([ptr(P[1]) for P in Ps], MAX_S, z), pad([ptr(P[2]) for P in Ps], MAX_S, z), pad(Int32[], MAX_S, Int32(0)),
            z, Float32(min_depth), Float32(max_depth), pad(Float32[], MAX_L, 0f0), 1f0, Int32(0), z,
            pad([gd], MAX_L, z), pad(gR, MAX_S, z), pad(gt, MAX_S, z), pad(P32[], MAX_S, z), pad(P32[], MAX_S, z), z, z, Int32(0), CuPtr{Int32}(0), Int32(0))
end
function rrule(::typeof(warp), disp::CuF, x::CuF, Ps, backprojections, projections, invKs::CuF, Ks::CuF; min_depth, max_depth, source_ids)
    outs = warp(disp, x, Ps, backprojections, projections, invKs, Ks; min_depth, max_depth, source_ids)
    function pb(Δ)
        gouts = [CuF(unthunk(d)) for d in unthunk(Δ)]
        gd = similar(disp); gR = [similar(P[1]) for P in Ps]; gt = [similar(P[2]) for P in Ps]
        desc = Ref(_warp_desc(disp, x, Ps, invKs, Ks, min_depth, max_depth, source_ids, (gd, gR, gt)))
        GC.@preserve disp x Ps invKs Ks gouts gd gR gt begin
            check(ccall((:md2_warp_bwd, LIB), Cint, (Ptr{Cvoid}, Ptr{VslDesc}, Ptr{P32}, Ptr{Cvoid}), ctx(), desc, [ptr(g) for g in gouts], stream()))
        end
        NoTangent(), gd, NoTangent(), [(r, t) for (r, t) in zip(gR, gt)],        # Ps is a Vector of (R, t) tuples
        NoTangent(), NoTangent(), NoTangent(), NoTangent()
    end
    outs, pb
end

"""
`slow_depth` (src/simple_depth.jl:1-62) for a Float32 triplet on the GPU: a METHOD of the reference's generic.  The 500
ADAM(3e-4) iterations over (disparity, 2 poses) run as a device-resident loop (`md2_slow_depth`: four launches per
iteration replayed from a CUDA graph); the host is involved only every `log_step` iterations, where the reference writes
its PNG and prints the poses.
"""
function slow_depth(x::CuArray{Float32, 5}, ssim, backprojections, projections, invKs::CuF, Ks::CuF, transfer;
                    target_id, source_ids, min_depth, max_depth, log_dir)
    W, H, C, Lf, N = size(x); S = length(source_ids)
    disp = CUDA.fill(0.5f0, W, H, 1, N)                                            # src/simple_depth.jl:8
    rvecs = [CuArray(repeat(Float32[0, 0, 0.01], 1, N)) for _ in 1:S]              # :9-13
    tvecs = [CUDA.zeros(Float32, 3, 1, N) for _ in 1:S]
    loss = CUDA.zeros(Float32, 1); gd = similar(disp); gr = similar.(rvecs); gt = similar.(tvecs)
    state = CUDA.zeros(Float32, 2 * (W * H * N + 6 * N * S)); clock = CUDA.zeros(Int64, 2)
    iters, log_step = 500, 5
    history = CUDA.zeros(Float32, iters)
    fs = Int64(W * H * C * Lf); z = P32(0)
    desc = Ref(VslDesc(W, H, N, C, S, 1, frameptr(x, target_id), fs,
        pad([frameptr(x, i) for i in source_ids], MAX_S, z), pad(fill(fs, S), MAX_S, Int64(0)),
        pad([ptr(disp)], MAX_L, z), pad(Int32[W], MAX_L, Int32(0)), pad(Int32[H], MAX_L, Int32(0)), ptr(Ks), ptr(invKs), Int32(1),
        pad(ptr.(rvecs), MAX_S, z), pad(ptr.(tvecs), MAX_S, z), pad(Int32[i < target_id for i in source_ids], MAX_S, Int32(0)), z,
        Float32(min_depth), Float32(max_depth), pad(Float32[1], MAX_L, 0f0), 1f0, Int32(0), ptr(loss),
        pad([ptr(gd)], MAX_L, z), pad(ptr.(gr), MAX_S, z), pad(ptr.(gt), MAX_S, z), pad(P32[], MAX_S, z),
        pad(P32[], MAX_S, z), z, z, Int32(0), CuPtr{Int32}(0), Int32(0)))
    done = 0
    GC.@preserve x disp rvecs tvecs loss gd gr gt state clock history Ks invKs begin
        while done < iters
            nxt = done == 0 ? 1 : min(iters, (done ÷ log_step + 1) * log_step)      # logs on iteration 1 and every 5th (:23)
            check(ccall((:md2_slow_depth, LIB), Cint,
                        (Ptr{Cvoid}, Ptr{VslDesc}, Cint, Cfloat, Cfloat, Cfloat, Cfloat, P32, CuPtr{Int64}, P32, Int64, Ptr{Cvoid}),
                        ctx(), desc, nxt - done, 3f-4, 0.9f0, 0.999f0, 1f-8, state, clock, history, iters, stream()))
            done = nxt
            save_disparity(reshape(Array(disp), (W, H)), joinpath(log_dir, "d-$done.png"))   # :47-49
            println(done, " ", mean(Array(disp)))
            for s in 1:S
                println("p$s.rvec, p$s.tvec = ", (Array(rvecs[s]), Array(tvecs[s])))
            end
        end
    end
    disp, [Pose(r, t) for (r, t) in zip(rvecs, tvecs)], Array(history)
end

# `warp` is the only NEW name (the reference calls it and never defines it): `using .B200: warp` in Monodepth.jl.
# view_synthesis_loss / vsl_fwdbwd / vsl_fwdbwd_host! are this binding's own additions.
export warp, view_synthesis_loss, vsl_fwdbwd, vsl_fwdbwd_host!, vsl_host_wait

end # module B200
