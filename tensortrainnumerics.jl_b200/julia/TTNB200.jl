# TTNB200.jl — thin `ccall` shim that routes TensorTrainNumerics.jl's hot-path methods to libttn_b200.so.
#
# Usage (after `using TensorTrainNumerics`):
#     include("TTNB200.jl"); using .TTNB200; TTNB200.init!(device = 0)
#     y = TTNB200.apply(A, x)                          # A * x                     src/tt_operations.jl:101
#     TTNB200.tt_compress!(ψ, 64; truncerr = 0.0)      # tt_compress!              src/tt_tools.jl:772
#     x = TTNB200.als_linsolve(A, b, x0; sweep_count = 4)                          # src/solvers/als.jl:161
#     E, ψ, r_hist = TTNB200.dmrg_eigsolve(H, ψ0; sweep_schedule = [2], rmax_schedule = [64])   # dmrg.jl:501
# `TTNB200.override!()` re-points the exported reference methods (`*`, `orthogonalize`, `tt_compress!`,
# `als_linsolve`, `mals_linsolve`, `dmrg_*`, `tdvp`, `tdvp2`) at these implementations.
#
# This file cannot be exercised in the build container (no Julia binary); it is kept deliberately thin — every call
# is (1) upload the cores, (2) one C-ABI call, (3) download — and the Python mirror in ../api.py drives the identical
# ABI under test, so the only untested code here is the marshalling below.
module TTNB200

using TensorTrainNumerics
import TensorTrainNumerics: TTvector, TToperator

const LIB = Ref{String}(joinpath(@__DIR__, "..", "libttn_b200.so"))
const F64, C128 = Cint(0), Cint(1)

struct TTNError <: Exception
    code::Int
    msg::String
end

function check(status::Cint)
    status == 0 && return nothing
    msg = unsafe_string(ccall((:ttn_last_error, LIB[]), Cstring, ()))
    # status -> the exception the reference throws at the same place (include/ttn_b200.h)
    status == 1 && throw(AssertionError(msg))        # "Incompatible dimensions"      tt_operations.jl:11,102
    status == 2 && throw(AssertionError(msg))        # sweeps >= 1, k in 1:N-1         tt_tools.jl:744,773
    status == 3 && throw(DimensionMismatch(msg))     # "Impossible orthogonalization"  tt_tools.jl:513
    status == 4 && throw(AssertionError(msg))        # "Sweep schedule error"          dmrg.jl:513
    throw(ErrorException("libttn_b200: $msg (status $status)"))
end

init!(; device::Integer = 0) = check(ccall((:ttn_init, LIB[]), Cint, (Cint,), device))

dtype_code(::Type{Float64}) = F64
dtype_code(::Type{ComplexF64}) = C128

# ---- containers ------------------------------------------------------------------------------------------------
mutable struct DevTT
    h::Ptr{Cvoid}
    function DevTT(h)
        x = new(h)
        finalizer(y -> ccall((:ttn_ttv_free, LIB[]), Cint, (Ptr{Cvoid},), y.h), x)
        return x
    end
end
mutable struct DevTTO
    h::Ptr{Cvoid}
    function DevTTO(h)
        x = new(h)
        finalizer(y -> ccall((:ttn_tto_free, LIB[]), Cint, (Ptr{Cvoid},), y.h), x)
        return x
    end
end

function upload(x::TTvector{T, M}) where {T <: Union{Float64, ComplexF64}, M}
    d = x.N
    dims = collect(Int64, x.ttv_dims)
    rks = collect(Int64, x.ttv_rks)
    ot = collect(Int64, x.ttv_ot)
    cores = [pointer(c) for c in x.ttv_vec]            # dense column-major (n, r_l, r_r): src/tt_tools.jl:25
    out = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve x check(ccall((:ttn_ttv_upload, LIB[]), Cint,
        (Cint, Cint, Ptr{Int64}, Ptr{Int64}, Ptr{Int64}, Ptr{Ptr{Cvoid}}, Cint, Ptr{Ptr{Cvoid}}),
        dtype_code(T), d, dims, rks, ot, cores, 1, out))
    return DevTT(out[])
end

function upload(A::TToperator{T, M}) where {T <: Union{Float64, ComplexF64}, M}
    d = A.N
    dims = collect(Int64, A.tto_dims)
    rks = collect(Int64, A.tto_rks)
    cores = [pointer(c) for c in A.tto_vec]            # (n, n, R_l, R_r): src/tt_tools.jl:50
    out = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve A check(ccall((:ttn_tto_upload, LIB[]), Cint,
        (Cint, Cint, Ptr{Int64}, Ptr{Int64}, Ptr{Ptr{Cvoid}}, Ptr{Ptr{Cvoid}}),
        dtype_code(T), d, dims, rks, cores, out))
    return DevTTO(out[])
end

function download(A::DevTTO)
    dt, d = Ref{Cint}(0), Ref{Cint}(0)
    check(ccall((:ttn_tto_info, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cint}, Ptr{Cint}), A.h, dt, d))
    N = Int(d[])
    T = dt[] == F64 ? Float64 : ComplexF64
    dims, rks = zeros(Int64, N), zeros(Int64, N + 1)
    check(ccall((:ttn_tto_dims, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Int64}), A.h, dims))
    check(ccall((:ttn_tto_ranks, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Int64}), A.h, rks))
    vec = [zeros(T, dims[k], dims[k], rks[k], rks[k + 1]) for k in 1:N]
    cores = [pointer(c) for c in vec]
    GC.@preserve vec check(ccall((:ttn_tto_download, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Ptr{Cvoid}}), A.h, cores))
    return TToperator{T, N}(N, vec, Tuple(dims), rks, zeros(Int64, N))
end

function download(x::DevTT)
    dt, d, b = Ref{Cint}(0), Ref{Cint}(0), Ref{Cint}(0)
    check(ccall((:ttn_ttv_info, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cint}, Ptr{Cint}, Ptr{Cint}), x.h, dt, d, b))
    N = Int(d[])
    T = dt[] == F64 ? Float64 : ComplexF64
    dims, rks, ot = zeros(Int64, N), zeros(Int64, N + 1), zeros(Int64, N)
    check(ccall((:ttn_ttv_dims, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Int64}), x.h, dims))
    check(ccall((:ttn_ttv_ranks, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Int64}), x.h, rks))
    check(ccall((:ttn_ttv_ot, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Int64}), x.h, ot))
    vec = [Array{T, 3}(undef, dims[k], rks[k], rks[k + 1]) for k in 1:N]
    ptrs = [pointer(c) for c in vec]
    GC.@preserve vec check(ccall((:ttn_ttv_download, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Ptr{Cvoid}}), x.h, ptrs))
    return TTvector{T, N}(N, vec, Tuple(dims), rks, ot)
end

# ---- TT algebra ------------------------------------------------------------------------------------------------
function apply(A::TToperator{T}, x::TTvector{T}) where {T}
    Ad, xd = upload(A), upload(x)
    out = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:ttn_apply, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Ptr{Cvoid}}), Ad.h, xd.h, out))
    return download(DevTT(out[]))
end

function dot(a::TTvector{T}, b::TTvector{T}) where {T}
    ad, bd = upload(a), upload(b)
    buf = zeros(Float64, 2)
    check(ccall((:ttn_dot, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}), ad.h, bd.h, buf))
    return T <: Real ? buf[1] : complex(buf[1], buf[2])
end

function orthogonalize(x::TTvector; i::Int = 1)
    xd = upload(x)
    out = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:ttn_orthogonalize, LIB[]), Cint, (Ptr{Cvoid}, Cint, Ptr{Ptr{Cvoid}}), xd.h, i, out))
    return download(DevTT(out[]))
end

function tt_compress!(ψ::TTvector, max_bond::Int; truncerr::Real = 0.0, sweeps::Int = 1, verbose::Bool = false)
    xd = upload(ψ)
    check(ccall((:ttn_compress, LIB[]), Cint, (Ptr{Cvoid}, Int64, Float64, Cint, Ptr{Float64}, Int64),
                xd.h, max_bond, truncerr, sweeps, C_NULL, 0))
    y = download(xd)
    # element-wise writes into the SAME `ttv_vec` / `ttv_rks` vectors, as src/tt_tools.jl:754-767 does: the QTTvector method
    # (src/qtt_tools.jl:783-786) relies on `TTvector(q)` sharing those vectors with `q`; ttv_ot stays untouched
    for k in 1:ψ.N
        ψ.ttv_vec[k] = y.ttv_vec[k]
    end
    ψ.ttv_rks .= y.ttv_rks
    return ψ
end

# `tt_compress!(A * x, max_bond; ...)` as ONE device call: the product cores of `A * x` are consumed by the first rounding pass
# without ever being written to memory (ttn_apply_compress; csrc/tt.cu).  A maintainer who wants the fusion behind the
# reference's own syntax makes `A * x` return a lazy `TTProduct(A, x)` and adds the method `tt_compress!(p::TTProduct, max_bond; ...)`
# that calls this function (every other consumer of a TTProduct materialises it with `apply`).
function apply_compress(A::TToperator{T}, x::TTvector{T}, max_bond::Int; truncerr::Real = 0.0, sweeps::Int = 1) where {T}
    Ad, xd = upload(A), upload(x)
    out = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:ttn_apply_compress, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Float64, Cint, Ptr{Float64}, Int64, Ptr{Ptr{Cvoid}}),
                Ad.h, xd.h, max_bond, truncerr, sweeps, C_NULL, 0, out))
    return download(DevTT(out[]))
end

# run-time switches of the library ("gram_compress", "gram_jacobi_min", "gemm_bulk", "gemm_thin", "reset_flops")
set_option!(key::AbstractString, value::Real) = check(ccall((:ttn_set_option, LIB[]), Cint, (Cstring, Float64), key, value))
function get_option(key::AbstractString)
    v = Ref{Float64}(0.0)
    check(ccall((:ttn_get_option, LIB[]), Cint, (Cstring, Ptr{Float64}), key, v))
    return v[]
end

# ---- site surgery (the other two-site-SVD users) -----------------------------------------------------------------------
const NO_CAP = Int64(1) << 62

# hadamard_ttm(x, y; tol, rmax)                                   src/tt_operations.jl:399-422
function hadamard_ttm(x::TTvector{T, N}, y::TTvector{T, N}; tol::Float64 = 1.0e-14, rmax::Int = typemax(Int)) where {T, N}
    @assert x.ttv_dims == y.ttv_dims "Incompatible TT dimensions"
    d = x.N
    cores = vcat([copy(c) for c in x.ttv_vec], [permutedims(y.ttv_vec[d + 1 - k], (1, 3, 2)) for k in 1:d])
    rks = vcat(collect(x.ttv_rks), reverse(collect(y.ttv_rks))[2:end])
    dims = (x.ttv_dims..., reverse(y.ttv_dims)...)
    z = upload(TTvector{T, 2d}(2d, cores, dims, rks, zeros(Int64, 2d)))
    cap = rmax >= NO_CAP ? NO_CAP : Int64(rmax)
    for iter in 1:d
        for j in d:-1:(d - iter + 2)                              # _ttm_swap!, :366-383
            check(ccall((:ttn_swap_sites, LIB[]), Cint, (Ptr{Cvoid}, Cint, Cint, Int64, Float64), z.h, j, 1, cap, tol))
        end
        check(ccall((:ttn_merge_sites_diag, LIB[]), Cint, (Ptr{Cvoid}, Cint), z.h, d - iter + 1))   # _ttm_contract!, :385-397
    end
    return download(z)
end

# the swap loop of reorder(q::QTTvector, new_ordering; threshold)  src/qtt_tools.jl:758-765
function apply_swaps(x::TTvector, swaps::Vector{Int}; threshold::Real = 0.0)
    xd = upload(x)
    for k in swaps
        check(ccall((:ttn_swap_sites, LIB[]), Cint, (Ptr{Cvoid}, Cint, Cint, Int64, Float64), xd.h, k, 0, NO_CAP, threshold))
    end
    return download(xd)
end

# to_qtt(tt, split_dims; threshold)                               src/qtt_tools.jl:254-310
function to_qtt(tt::TTvector, split_dims::Vector{Vector{Int}}; threshold::Float64 = 0.0)
    @assert length(split_dims) == tt.N "split_dims must have one entry per TT core"
    xd = upload(tt)
    site = 1
    for sd in split_dims
        for s in sd[1:(end - 1)]
            check(ccall((:ttn_split_site, LIB[]), Cint, (Ptr{Cvoid}, Cint, Int64, Cint, Int64, Float64), xd.h, site, s, 0, NO_CAP, threshold))
            site += 1
        end
        site += 1
    end
    return download(xd)
end

# ---- solvers ---------------------------------------------------------------------------------------------------
# mirrors `ttn_solver_params` (include/ttn_b200.h)
struct SolverParams
    N::Cint
    tol::Cdouble
    sweep_schedule::Ptr{Int64}
    n_sweep_schedule::Cint
    rmax_schedule::Ptr{Int64}
    n_rmax_schedule::Cint
    rmax::Int64
    sweep_count::Cint
    it_solver::Cint
    linsolv_maxiter::Cint
    linsolv_tol::Cdouble
    itslv_thresh::Cint
    krylovdim::Cint
    symmetrize::Cint
end

function params(; N = 2, tol = 1.0e-12, sweep_schedule = Int64[], rmax_schedule = Int64[], rmax = 0, sweep_count = 2,
                it_solver = false, linsolv_maxiter = 200, linsolv_tol = 1.0e-6, itslv_thresh = 256, krylovdim = 30,
                symmetrize = false)
    ss, rs = collect(Int64, sweep_schedule), collect(Int64, rmax_schedule)
    p = SolverParams(N, tol, pointer(ss), length(ss), pointer(rs), length(rs), rmax, sweep_count, it_solver,
                     linsolv_maxiter, linsolv_tol, itslv_thresh, krylovdim, symmetrize)
    return p, (ss, rs)          # keep the schedule vectors alive for the duration of the call
end

function _linsolve(sym::Symbol, A, b, x0, p, keep; return_info = false)
    Ad, bd, xd = upload(A), upload(b), upload(x0)
    out, res = Ref{Ptr{Cvoid}}(C_NULL), Ref{Float64}(0.0)
    GC.@preserve keep check(ccall((sym, LIB[]), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ref{SolverParams}, Ptr{Ptr{Cvoid}}, Ptr{Float64}),
        Ad.h, bd.h, xd.h, Ref(p), out, return_info ? res : C_NULL))
    x = download(DevTT(out[]))
    return return_info ? (x, (; residual = res[])) : x
end

function als_linsolve(A, b, tt_start; sweep_count = 2, it_solver = false, r_itsolver = 5000, return_info = false)
    p, keep = params(; sweep_count)
    return _linsolve(:ttn_als_linsolve, A, b, tt_start, p, keep; return_info)
end

function mals_linsolve(A, b, tt_start; tol = 1.0e-12, rmax = round(Int, sqrt(prod(tt_start.ttv_dims))), return_info = false)
    p, keep = params(; tol, rmax)
    return _linsolve(:ttn_mals_linsolve, A, b, tt_start, p, keep; return_info)
end

function dmrg_linsolve(A, b, tt_start; sweep_count = 2, N = 2, tol = 1.0e-12, sweep_schedule = [2],
                       rmax_schedule = [isqrt(prod(tt_start.ttv_dims))], it_solver = true, linsolv_maxiter = 200,
                       linsolv_tol = max(sqrt(tol), 1.0e-8), itslv_thresh = 256, return_info = false)
    p, keep = params(; N, tol, sweep_schedule, rmax_schedule, linsolv_maxiter, linsolv_tol, itslv_thresh, symmetrize = true)
    return _linsolve(:ttn_dmrg_linsolve, A, b, tt_start, p, keep; return_info)
end

function _eigsolve(sym::Symbol, A, x0, p, keep, cap)
    Ad, xd = upload(A), upload(x0)
    out, nE = Ref{Ptr{Cvoid}}(C_NULL), Ref{Cint}(0)
    E, rh = zeros(Float64, cap), zeros(Int64, cap)
    GC.@preserve keep check(ccall((sym, LIB[]), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ref{SolverParams}, Ptr{Ptr{Cvoid}}, Ptr{Float64}, Ptr{Int64}, Cint, Ptr{Cint}),
        Ad.h, xd.h, Ref(p), out, E, rh, cap, nE))
    return E[1:nE[]], download(DevTT(out[])), rh[1:nE[]]
end

# als_eigsolve(A, tt_start; sweep_schedule, rmax_schedule, ...)    src/solvers/als.jl:251-321 (noise_schedule == 0 only)
function als_eigsolve(A, tt_start; sweep_schedule = [2], rmax_schedule = [maximum(tt_start.ttv_rks)],
                      noise_schedule = zeros(length(rmax_schedule)), it_solver = false, itslv_thresh = 1024, maxiter = 200,
                      linsolv_tol = 1.0e-8)
    all(iszero, noise_schedule) || error("noise_schedule != 0 draws from the host RNG and is not on the device path")
    p, keep = params(; sweep_schedule, rmax_schedule, linsolv_maxiter = maxiter, linsolv_tol, krylovdim = 30)
    Ad, xd = upload(A), upload(tt_start)
    cap = 2 * tt_start.N * (sweep_schedule[end] + 1) + 8
    out, nE, E = Ref{Ptr{Cvoid}}(C_NULL), Ref{Cint}(0), zeros(Float64, cap)
    GC.@preserve keep check(ccall((:ttn_als_eigsolve, LIB[]), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ref{SolverParams}, Ptr{Ptr{Cvoid}}, Ptr{Float64}, Cint, Ptr{Cint}),
        Ad.h, xd.h, Ref(p), out, E, cap, nE))
    return E[1:nE[]], download(DevTT(out[]))
end

# als_gen_eigsolv(A, S, tt_start; ...)                            src/solvers/als.jl:344-440
function als_gen_eigsolv(A, S, tt_start; sweep_schedule = [2], rmax_schedule = [maximum(tt_start.ttv_rks)], tol = 1.0e-10,
                         it_solver = false, itslv_thresh = 2500)
    p, keep = params(; sweep_schedule, rmax_schedule, linsolv_maxiter = 500, linsolv_tol = 1.0e-12, krylovdim = 40)
    Ad, Sd, xd = upload(A), upload(S), upload(tt_start)
    cap = 2 * tt_start.N * (sweep_schedule[end] + 1) + 8
    out, nE, E = Ref{Ptr{Cvoid}}(C_NULL), Ref{Cint}(0), zeros(Float64, cap)
    GC.@preserve keep check(ccall((:ttn_als_gen_eigsolv, LIB[]), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ref{SolverParams}, Ptr{Ptr{Cvoid}}, Ptr{Float64}, Cint, Ptr{Cint}),
        Ad.h, Sd.h, xd.h, Ref(p), out, E, cap, nE))
    return E[1:nE[]], download(DevTT(out[]))
end

function dmrg_eigsolve(A, tt_start; N = 2, tol = 1.0e-12, sweep_schedule = [2],
                       rmax_schedule = [isqrt(prod(tt_start.ttv_dims))], it_solver = false, linsolv_maxiter = 200,
                       linsolv_tol = max(sqrt(tol), 1.0e-8), itslv_thresh = 256)
    @assert length(rmax_schedule) == length(sweep_schedule) "Sweep schedule error"
    p, keep = params(; N, tol, sweep_schedule, rmax_schedule, linsolv_maxiter, linsolv_tol, itslv_thresh, symmetrize = true)
    return _eigsolve(:ttn_dmrg_eigsolve, A, tt_start, p, keep, 2 * A.N * (sweep_schedule[end] + 1) + 8)
end

function mals_eigsolve(A, tt_start; tol = 1.0e-12, sweep_schedule = [2],
                       rmax_schedule = [round(Int, sqrt(prod(tt_start.ttv_dims)))], it_solver = false,
                       linsolv_maxiter = 200, linsolv_tol = max(sqrt(tol), 1.0e-8), itslv_thresh = 256)
    @assert length(rmax_schedule) == length(sweep_schedule) "Sweep schedule error"
    p, keep = params(; tol, sweep_schedule, rmax_schedule, linsolv_maxiter, linsolv_tol, itslv_thresh)
    return _eigsolve(:ttn_mals_eigsolve, A, tt_start, p, keep, 2 * A.N * (sweep_schedule[end] + 1) + 8)
end

# mirrors `ttn_tdvp_params`
struct TdvpParams
    two_site::Cint
    steps::Ptr{Float64}
    n_steps::Cint
    normalize::Cint
    sweeps::Cint
    imaginary_time::Cint
    max_bond::Int64
    truncerr::Cdouble
    krylovdim::Cint
    krylov_tol::Cdouble
    krylov_maxiter::Cint
end

function _tdvp(two_site, H, u0, steps; normalize = true, sweeps = 1, max_bond = typemax(Int) >> 1, truncerr = 0.0,
               imaginary_time = false, krylovdim = 30, tol = 1.0e-12, maxiter = 100)
    Hd, ud = upload(H), upload(u0)
    st = collect(Float64, steps)
    p = TdvpParams(two_site, pointer(st), length(st), normalize, sweeps, imaginary_time, max_bond, truncerr, krylovdim, tol, maxiter)
    out = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve st check(ccall((:ttn_tdvp, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ref{TdvpParams}, Ptr{Ptr{Cvoid}}),
                                Hd.h, ud.h, Ref(p), out))
    return download(DevTT(out[]))
end
tdvp(H, u0, steps::Vector{Float64}; kwargs...) = _tdvp(0, H, u0, steps; kwargs...)
tdvp2(H, u0, steps::Vector{Float64}; kwargs...) = _tdvp(1, H, u0, steps; kwargs...)

"""Re-point the reference's exported hot-path methods at the B200 implementations."""
# ---- one bond problem sharded over the GPUs of a node (SURVEY.md section 8(e)); `allgather` is e.g. b -> MPI.Allgather(b, comm) ----
mutable struct ShardedMatvec
    h::Ptr{Cvoid}
    function ShardedMatvec(G::Array{T, 3}, Amid::Array{T, 4}, H::Array{T, 3}, rank::Int, nranks::Int, allgather) where {T <: Union{Float64, ComplexF64}}
        out = Ref{Ptr{Cvoid}}(C_NULL)
        GC.@preserve G Amid H check(ccall((:ttn_shard_matvec_create, LIB), Cint,
            (Cint, Cint, Cint, Cint, Cint, Cint, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Cint, Cint, Ptr{Ptr{Cvoid}}),
            T === Float64 ? 0 : 1, size(G, 1), size(H, 1), size(G, 2), size(H, 2), size(Amid, 2), G, Amid, H, rank, nranks, out))
        mv = new(out[])
        finalizer(m -> ccall((:ttn_shard_matvec_free, LIB), Cint, (Ptr{Cvoid},), m.h), mv)
        if nranks > 1
            mine = Vector{UInt8}(undef, 192)
            check(ccall((:ttn_shard_matvec_handles, LIB), Cint, (Ptr{Cvoid}, Ptr{UInt8}), mv.h, mine))
            all = allgather(mine)::Vector{UInt8}                  # nranks * 192 bytes in rank order
            check(ccall((:ttn_shard_matvec_bind, LIB), Cint, (Ptr{Cvoid}, Ptr{UInt8}), mv.h, all))
        end
        return mv
    end
end

"lowest eigenpair of the sharded effective operator; `x_dev` is a device pointer (start vector in, eigenvector out)"
function shard_eigsolve(mv::ShardedMatvec, x_dev::Ptr{Cvoid}; krylovdim = 8, maxiter = 1, tol = 1.0e-10)
    theta = Ref{Cdouble}(0.0); nmv = Ref{Cint}(0)
    check(ccall((:ttn_shard_eigsolve, LIB), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Cint, Cint, Cdouble, Ptr{Cdouble}, Ptr{Cint}),
                mv.h, x_dev, krylovdim, maxiter, tol, theta, nmv))
    return theta[], Int(nmv[])
end

function override!()
    @eval TensorTrainNumerics begin
        Base.:*(A::TToperator{T, N}, v::TTvector{T, N}) where {T <: Union{Float64, ComplexF64}, N} = $(apply)(A, v)
        orthogonalize(x::TTvector{T, N}; i = 1::Int) where {T <: Union{Float64, ComplexF64}, N} = $(orthogonalize)(x; i = i)
        tt_compress!(ψ::TTvector{T, N}, max_bond::Int; kwargs...) where {T <: Union{Float64, ComplexF64}, N} =
            $(tt_compress!)(ψ, max_bond; kwargs...)
        als_linsolve(A::TToperator, b::TTvector, x0::TTvector; kwargs...) = $(als_linsolve)(A, b, x0; kwargs...)
        mals_linsolve(A::TToperator, b::TTvector, x0::TTvector; kwargs...) = $(mals_linsolve)(A, b, x0; kwargs...)
        dmrg_linsolve(A::TToperator, b::TTvector, x0::TTvector; kwargs...) = $(dmrg_linsolve)(A, b, x0; kwargs...)
        als_eigsolve(A::TToperator, x0::TTvector; kwargs...) = $(als_eigsolve)(A, x0; kwargs...)
        als_gen_eigsolv(A::TToperator, S::TToperator, x0::TTvector; kwargs...) = $(als_gen_eigsolv)(A, S, x0; kwargs...)
        dmrg_eigsolve(A::TToperator, x0::TTvector; kwargs...) = $(dmrg_eigsolve)(A, x0; kwargs...)
        mals_eigsolve(A::TToperator, x0::TTvector; kwargs...) = $(mals_eigsolve)(A, x0; kwargs...)
        tdvp(H::TToperator, u0::TTvector, steps::Vector{Float64}; kwargs...) = $(tdvp)(H, u0, steps; kwargs...)
        tdvp2(H::TToperator, u0::TTvector, steps::Vector{Float64}; kwargs...) = $(tdvp2)(H, u0, steps; kwargs...)
        hadamard_ttm(x::TTvector{T, N}, y::TTvector{T, N}; kwargs...) where {T <: Union{Float64, ComplexF64}, N} =
            $(hadamard_ttm)(x, y; kwargs...)
        to_qtt(tt::TTvector{T, N}, split_dims::Vector{Vector{Int}}; kwargs...) where {T <: Union{Float64, ComplexF64}, N} =
            $(to_qtt)(tt, split_dims; kwargs...)
        # QTTvector / QTToperator methods (src/qtt_tools.jl:526-534, 590-598, 783-786) delegate to the TTvector / TToperator
        # methods re-pointed above and re-wrap the result themselves, so they need no entries of their own; `reorder`
        # (src/qtt_tools.jl:731-774) keeps its permutation logic and only its swap loop moves to the device:
        function reorder(q::QTTvector, new_ordering::Symbol; threshold::Real = 0.0)
            @assert new_ordering ∈ (:interleaved, :serial) "ordering must be :interleaved or :serial"
            q.ordering == new_ordering && return copy(q)
            perm = zeros(Int, q.N)
            for d in 1:q.n_dims, b in 0:(q.bits_per_dim - 1)
                if q.ordering == :serial
                    perm[(d - 1) * q.bits_per_dim + b + 1] = b * q.n_dims + (d - 1)
                else
                    perm[b * q.n_dims + (d - 1) + 1] = (d - 1) * q.bits_per_dim + b
                end
            end
            y = $(apply_swaps)(TTvector(q), _bubble_sort_swaps(perm); threshold = threshold)
            return QTTvector(y, q.n_dims, q.bits_per_dim, new_ordering)
        end
    end
    return nothing
end

end # module
