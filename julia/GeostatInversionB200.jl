# GeostatInversionB200.jl -- `ccall` shim over libgsi_b200.so (include/gsi_b200.h).
#
# UNTESTED HERE: Julia is not installed in the build image; this file is a mechanical
# transcription of the header (the same table the tested Python `ctypes` host uses,
# geostatinversion.jl_b200/_lib.py).  tests/test_julia_shim.py parses every `ccall` below and
# checks its symbol, return type, argument count and argument classes against the header.
# It keeps the reference's call surface (SURVEY.md §8b):
#   RandMatFact.randsvd(A, K, p, q), rangefinder(A, l, q), rangefinder(A; epsilon, r),
#   eig_nystrom(A, Q), getxis(Q, numxis, p, q, seed), getxis(samplefield, numfields, numxis, p, q, seed),
#   getxis(Val{:iwantfields}, ...), pcgalsqr / pcgadirect / pcga / rga with the reference's
#   positional and keyword arguments,
# plus covsolve(C, B; rtol, maxiter, rank, seed), the dense factor covchol(C) with covchol_solve / covchol_logdet /
# covchol_variance, krige(...; method = :cg | :cholesky, variance), covchol(C; diag), covchol_simulate, the
# conditional / unconditional simulate(...), the likelihood covloglik(C, y; drift, reml, grad) and cross-validation
# covchol_crossval(f, y; drift, groups) on the kernel-covariance operators (new),
# for A::Matrix{Float64}, A::KernelCovMatrix (new), A::KernelCrossCovMatrix (new, not symmetric) and
# A::LowRankCovMatrix, whose method set is
# the one the reference's LowRankCovMatrix provides (src/lowrank.jl:38-60,115-139):
#   size(A), size(A, i), A', A * Matrix, A * Vector, Adjoint{Matrix} * A.
module GeostatInversionB200

import Random
import LinearAlgebra
import Distributed
import SparseArrays

const LIB = get(ENV, "GSI_B200_LIB", joinpath(@__DIR__, "..", "geostatinversion.jl_b200", "lib", "libgsi_b200.so"))

const GSI_LAYOUT_TALL = Int32(0)
const GSI_LAYOUT_COLMAJOR = Int32(1)
const GSI_NORMALISER_LU_REF = Int32(0)
const GSI_KERNEL_EXPONENTIAL = Int32(0)
const GSI_KERNEL_GAUSSIAN = Int32(1)
const GSI_KERNEL_POWERLAW = Int32(2)
const GSI_KERNEL_MATERN32 = Int32(3)
const GSI_KERNEL_MATERN52 = Int32(4)
const GSI_KERNEL_SPHERICAL = Int32(5)

lasterror() = unsafe_string(ccall((:gsi_last_error_string, LIB), Cstring, ()))

"status code of include/gsi_b200.h -> the exception the reference's own code path would raise"
function check(status::Int32)
	status == 0 && return nothing
	msg = lasterror()
	status == 1 && throw(ArgumentError(msg))                      # GSI_ERR_INVALID_ARGUMENT
	status == 2 && throw(DimensionMismatch(msg))
	if status == 3                                                # lu(...; check=true), RandMatFact.jl:60,68,72
		m = match(r"SingularException\((\d+)\)", msg)
		throw(LinearAlgebra.SingularException(m === nothing ? 0 : parse(Int, m.captures[1])))
	end
	if status == 4                                                # cholesky in eig_nystrom, RandMatFact.jl:95
		m = match(r"PosDefException\((-?\d+)\)", msg)
		throw(LinearAlgebra.PosDefException(m === nothing ? 0 : parse(Int, m.captures[1])))
	end
	status == 9 && error(msg)       # "parameter numiterations should be positive, but numiterations=$q", RandMatFact.jl:63
	error(msg)                      # CUDA / NCCL / no device / unsupported / no convergence
end

mutable struct Context
	h::Ptr{Cvoid}
	rank::Int
	world::Int
	function Context(device::Integer=0; rank::Integer=0, world::Integer=1, uid::Vector{UInt8}=UInt8[])
		world > 1 && length(uid) != 128 && throw(ArgumentError("world > 1 needs the 128-byte id of uniqueid() from rank 0"))
		out = Ref{Ptr{Cvoid}}(C_NULL)
		GC.@preserve uid check(ccall((:gsi_ctx_create, LIB), Int32, (Int32, Int32, Int32, Ptr{UInt8}, Ref{Ptr{Cvoid}}),
			device, rank, world, world > 1 ? pointer(uid) : Ptr{UInt8}(C_NULL), out))
		ctx = new(out[], rank, world)
		finalizer(c->ccall((:gsi_ctx_destroy, LIB), Int32, (Ptr{Cvoid},), c.h), ctx)
		return ctx
	end
end

"128-byte NCCL id: call on rank 0, send to the other workers, pass as `uid` to every `Context`"
function uniqueid()
	id = Vector{UInt8}(undef, 128)
	GC.@preserve id check(ccall((:gsi_comm_unique_id, LIB), Int32, (Ptr{UInt8},), id))
	return id
end

sync(ctx::Context) = check(ccall((:gsi_ctx_sync, LIB), Int32, (Ptr{Cvoid},), ctx.h))

"contiguous row block (1-based range) of worker `rank` (0-based) out of `world`: blocks are multiples of 64 rows"
function partitionrows(n::Integer, world::Integer, rank::Integer; align::Integer=64)
	per = cld(cld(n, world), align) * align
	r0 = min(n, rank * per)
	r1 = min(n, r0 + per)
	return (r0 + 1):r1
end

# tuning knobs of include/gsi_b200.h (gsi_ctx_set_option), e.g. setoption!(ctx, "kcov.window", 8)
setoption!(ctx::Context, name::AbstractString, value::Integer) =
	check(ccall((:gsi_ctx_set_option, LIB), Int32, (Ptr{Cvoid}, Cstring, Int64), ctx.h, name, value))
function getoption(ctx::Context, name::AbstractString)
	v = Ref{Int64}(0)
	check(ccall((:gsi_ctx_get_option, LIB), Int32, (Ptr{Cvoid}, Cstring, Ref{Int64}), ctx.h, name, v))
	return v[]
end

const defaultctx = Ref{Union{Nothing, Context}}(nothing)
context() = (defaultctx[] === nothing && (defaultctx[] = Context()); defaultctx[])
setcontext!(ctx::Context) = (defaultctx[] = ctx)

mutable struct DeviceMatrix
	h::Ptr{Cvoid}
	rows::Int
	cols::Int
	function DeviceMatrix(ctx::Context, layout::Int32, rows::Integer, cols::Integer)
		out = Ref{Ptr{Cvoid}}(C_NULL)
		check(ccall((:gsi_buf_alloc, LIB), Int32, (Ptr{Cvoid}, Int32, Int64, Int64, Ref{Ptr{Cvoid}}), ctx.h, layout, rows, cols, out))
		b = new(out[], rows, cols)
		finalizer(x->ccall((:gsi_buf_free, LIB), Int32, (Ptr{Cvoid},), x.h), b)    # idempotent, never throws
		return b
	end
end

function upload!(b::DeviceMatrix, A::Matrix{Float64})
	size(A) == (b.rows, b.cols) || throw(DimensionMismatch("upload!: host $(size(A)) vs device $((b.rows, b.cols))"))
	GC.@preserve A check(ccall((:gsi_buf_upload, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}, Int64), b.h, A, max(1, size(A, 1))))
	return b
end

function download(b::DeviceMatrix)
	A = Matrix{Float64}(undef, b.rows, b.cols)
	GC.@preserve A check(ccall((:gsi_buf_download, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}, Int64), b.h, A, max(1, b.rows)))
	return A
end

"Matrix{Float64} in page-locked host memory (gsi_host_alloc): `upload!` from it is a plain DMA.  Release with `freepinned`."
function pinnedmatrix(ctx::Context, rows::Integer, cols::Integer)
	out = Ref{Ptr{Cvoid}}(C_NULL)
	check(ccall((:gsi_host_alloc, LIB), Int32, (Ptr{Cvoid}, Int64, Ref{Ptr{Cvoid}}), ctx.h, 8 * max(1, rows * cols), out))
	return unsafe_wrap(Array, Ptr{Float64}(out[]), (Int(rows), Int(cols)); own=false)
end
freepinned(ctx::Context, A::Matrix{Float64}) = check(ccall((:gsi_host_free, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}), ctx.h, pointer(A)))

# One product pass handles at most 256 columns; wider host matrices go through in passes.  A TALL device
# iterate itself may be up to 1024 columns wide (the library runs its products in 256-column chunks).
const MAXCOLS = 256
const MAXWIDECOLS = 1024

abstract type Operator end
# `rows` = this worker's block of global rows (all rows on a single-GPU context)
mutable struct DenseOperator <: Operator; h::Ptr{Cvoid}; buf::DeviceMatrix; ctx::Context; rows::UnitRange{Int}; end
# nparams: the length of the likelihood gradient (covloglik), nstruct (1 + d) + 1
mutable struct KernelCovMatrix <: Operator; h::Ptr{Cvoid}; n::Int; ctx::Context; rows::UnitRange{Int}; nparams::Int; end
mutable struct LowRankCovMatrix <: Operator; h::Ptr{Cvoid}; buf::DeviceMatrix; ctx::Context; rows::UnitRange{Int}; end
# cross-covariance C(T, S): `rows` = this worker's block of target rows
mutable struct KernelCrossCovMatrix <: Operator; h::Ptr{Cvoid}; n::Int; ctx::Context; rows::UnitRange{Int}; end
issym(::DenseOperator) = false
issym(::KernelCrossCovMatrix) = false
issym(::Operator) = true

freeop(o) = ccall((:gsi_op_free, LIB), Int32, (Ptr{Cvoid},), o.h)

"""
Dense `A::Matrix` (src/GeostatInversion.jl:63).  Multi-GPU: pass this worker's row block
`A[rows, :]` together with `rows` and the global row count `m`.
"""
function DenseOperator(A::Matrix{Float64}; ctx::Context=context(), rows::UnitRange{Int}=1:size(A, 1), m::Integer=size(A, 1))
	length(rows) == size(A, 1) || throw(DimensionMismatch("DenseOperator: A must hold exactly the rows `rows`"))
	buf = upload!(DeviceMatrix(ctx, GSI_LAYOUT_COLMAJOR, size(A)...), A)
	out = Ref{Ptr{Cvoid}}(C_NULL)
	check(ccall((:gsi_op_dense, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int64, Ref{Ptr{Cvoid}}), ctx.h, buf.h, first(rows) - 1, m, out))
	op = DenseOperator(out[], buf, ctx, rows)
	finalizer(freeop, op)
	return op
end

"kind: 0 exponential, 1 gaussian, 2 powerlaw, 3 matern32, 4 matern52, 5 spherical (GSI_KERNEL_*; ell is the spherical
model's range); coords d x n; ell d.  Multi-GPU: `rows` = this worker's rows of C."
function KernelCovMatrix(kind::Integer, coords::Matrix{Float64}, ell::Vector{Float64}; sigma2=1.0, nugget=0.0, beta=1.0,
		ctx::Context=context(), rows::UnitRange{Int}=partitionrows(size(coords, 2), ctx.world, ctx.rank))
	d, n = size(coords)
	out = Ref{Ptr{Cvoid}}(C_NULL)
	GC.@preserve coords ell check(ccall((:gsi_op_kernelcov, LIB), Int32,
		(Ptr{Cvoid}, Int32, Int32, Int64, Ptr{Float64}, Ptr{Float64}, Float64, Float64, Float64, Int64, Int64, Ref{Ptr{Cvoid}}),
		ctx.h, kind, d, n, coords, ell, sigma2, nugget, beta, first(rows) - 1, length(rows), out))
	op = KernelCovMatrix(out[], n, ctx, rows, d + 2)
	finalizer(freeop, op)
	return op
end

"structured grid variant (same kinds): dims[1] fastest (Julia linear index), coordinates idx .* spacing"
function KernelCovGrid(kind::Integer, dims::Vector{Int}, spacing::Vector{Float64}, ell::Vector{Float64}; sigma2=1.0, nugget=0.0, beta=1.0,
		ctx::Context=context(), rows::UnitRange{Int}=partitionrows(prod(dims), ctx.world, ctx.rank))
	d = length(dims)
	n = prod(dims)
	out = Ref{Ptr{Cvoid}}(C_NULL)
	dims64 = Int64.(dims)
	GC.@preserve dims64 spacing ell check(ccall((:gsi_op_kernelcov_grid, LIB), Int32,
		(Ptr{Cvoid}, Int32, Int32, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Float64, Float64, Float64, Int64, Int64, Ref{Ptr{Cvoid}}),
		ctx.h, kind, d, dims64, spacing, ell, sigma2, nugget, beta, first(rows) - 1, length(rows), out))
	op = KernelCovMatrix(out[], n, ctx, rows, d + 2)
	finalizer(freeop, op)
	return op
end

"""Nested covariance model (gsi_op_kernelcov_model): C = sum_s sills[s] k_{kinds[s]} + nugget I, 1 to
GSI_MODEL_MAX_STRUCTURES structures.  ranges d x nstruct; rotations d x d x nstruct (u = R x, orthonormal) or
`nothing` (no rotation); betas (power law) or `nothing` (1)."""
function KernelCovModel(kinds::Vector{<:Integer}, sills::Vector{Float64}, ranges::Matrix{Float64}, coords::Matrix{Float64};
		rotations::Union{Nothing, Array{Float64, 3}}=nothing, betas::Union{Nothing, Vector{Float64}}=nothing, nugget=0.0,
		ctx::Context=context(), rows::UnitRange{Int}=partitionrows(size(coords, 2), ctx.world, ctx.rank))
	d, n = size(coords)
	kinds32 = Int32.(kinds)
	rot = rotations === nothing ? Ptr{Float64}(C_NULL) : pointer(rotations)
	bet = betas === nothing ? Ptr{Float64}(C_NULL) : pointer(betas)
	out = Ref{Ptr{Cvoid}}(C_NULL)
	GC.@preserve coords kinds32 sills ranges rotations betas check(ccall((:gsi_op_kernelcov_model, LIB), Int32,
		(Ptr{Cvoid}, Int32, Int64, Ptr{Float64}, Int32, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
		 Float64, Int64, Int64, Ref{Ptr{Cvoid}}),
		ctx.h, d, n, coords, length(kinds32), kinds32, sills, ranges, rot, bet, nugget, first(rows) - 1, length(rows), out))
	op = KernelCovMatrix(out[], n, ctx, rows, length(kinds) * (1 + d) + 1)
	finalizer(freeop, op)
	return op
end

"structured grid variant of KernelCovModel (the model is tabulated once per lattice offset)"
function KernelCovModelGrid(kinds::Vector{<:Integer}, sills::Vector{Float64}, ranges::Matrix{Float64}, dims::Vector{Int},
		spacing::Vector{Float64}; rotations::Union{Nothing, Array{Float64, 3}}=nothing,
		betas::Union{Nothing, Vector{Float64}}=nothing, nugget=0.0,
		ctx::Context=context(), rows::UnitRange{Int}=partitionrows(prod(dims), ctx.world, ctx.rank))
	d = length(dims)
	n = prod(dims)
	dims64 = Int64.(dims)
	kinds32 = Int32.(kinds)
	rot = rotations === nothing ? Ptr{Float64}(C_NULL) : pointer(rotations)
	bet = betas === nothing ? Ptr{Float64}(C_NULL) : pointer(betas)
	out = Ref{Ptr{Cvoid}}(C_NULL)
	GC.@preserve dims64 spacing kinds32 sills ranges rotations betas check(ccall((:gsi_op_kernelcov_model_grid, LIB), Int32,
		(Ptr{Cvoid}, Int32, Ptr{Int64}, Ptr{Float64}, Int32, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
		 Float64, Int64, Int64, Ref{Ptr{Cvoid}}),
		ctx.h, d, dims64, spacing, length(kinds32), kinds32, sills, ranges, rot, bet, nugget, first(rows) - 1, length(rows), out))
	op = KernelCovMatrix(out[], n, ctx, rows, length(kinds) * (1 + d) + 1)
	finalizer(freeop, op)
	return op
end

"""Cross-covariance C(T, S) of a nested model (gsi_op_kernelcov_cross) between targets d x m and sources d x n, no
nugget: kriging `C(T, S) * w`, `Q H' = C(grid, obs)`.  Model arguments as KernelCovModel.  Not symmetric: `A' * X` is
C(S, T) X (all n rows, summed over workers).  Multi-GPU: `rows` = this worker's target rows."""
function KernelCrossCov(kinds::Vector{<:Integer}, sills::Vector{Float64}, ranges::Matrix{Float64}, targets::Matrix{Float64},
		sources::Matrix{Float64}; rotations::Union{Nothing, Array{Float64, 3}}=nothing,
		betas::Union{Nothing, Vector{Float64}}=nothing,
		ctx::Context=context(), rows::UnitRange{Int}=partitionrows(size(targets, 2), ctx.world, ctx.rank))
	d, m = size(targets)
	size(sources, 1) == d || throw(DimensionMismatch("KernelCrossCov: targets are $d-D, sources $(size(sources, 1))-D"))
	n = size(sources, 2)
	kinds32 = Int32.(kinds)
	rot = rotations === nothing ? Ptr{Float64}(C_NULL) : pointer(rotations)
	bet = betas === nothing ? Ptr{Float64}(C_NULL) : pointer(betas)
	out = Ref{Ptr{Cvoid}}(C_NULL)
	GC.@preserve targets sources kinds32 sills ranges rotations betas check(ccall((:gsi_op_kernelcov_cross, LIB), Int32,
		(Ptr{Cvoid}, Int32, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Int32, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
		 Ptr{Float64}, Int64, Int64, Ref{Ptr{Cvoid}}),
		ctx.h, d, m, targets, n, sources, length(kinds32), kinds32, sills, ranges, rot, bet, first(rows) - 1, length(rows), out))
	op = KernelCrossCovMatrix(out[], n, ctx, rows)
	finalizer(freeop, op)
	return op
end

"""structured grid variant of KernelCrossCov: targets / sources are 1-based linear indices of grid nodes (dims[1]
fastest), `nothing` for every node in order"""
function KernelCrossCovGrid(kinds::Vector{<:Integer}, sills::Vector{Float64}, ranges::Matrix{Float64}, dims::Vector{Int},
		spacing::Vector{Float64}, targets::Union{Nothing, AbstractVector{<:Integer}}, sources::Union{Nothing, AbstractVector{<:Integer}};
		rotations::Union{Nothing, Array{Float64, 3}}=nothing, betas::Union{Nothing, Vector{Float64}}=nothing,
		ctx::Context=context(), rows::UnitRange{Int}=partitionrows(targets === nothing ? prod(dims) : length(targets), ctx.world, ctx.rank))
	d = length(dims)
	dims64 = Int64.(dims)
	tidx = targets === nothing ? nothing : Int64.(targets) .- 1                # 0-based for the library
	sidx = sources === nothing ? nothing : Int64.(sources) .- 1
	m = tidx === nothing ? prod(dims) : length(tidx)
	n = sidx === nothing ? prod(dims) : length(sidx)
	tp = tidx === nothing ? Ptr{Int64}(C_NULL) : pointer(tidx)
	sp = sidx === nothing ? Ptr{Int64}(C_NULL) : pointer(sidx)
	kinds32 = Int32.(kinds)
	rot = rotations === nothing ? Ptr{Float64}(C_NULL) : pointer(rotations)
	bet = betas === nothing ? Ptr{Float64}(C_NULL) : pointer(betas)
	out = Ref{Ptr{Cvoid}}(C_NULL)
	GC.@preserve dims64 spacing tidx sidx kinds32 sills ranges rotations betas check(ccall((:gsi_op_kernelcov_cross_grid, LIB), Int32,
		(Ptr{Cvoid}, Int32, Ptr{Int64}, Ptr{Float64}, Int64, Ptr{Int64}, Int64, Ptr{Int64}, Int32, Ptr{Int32}, Ptr{Float64},
		 Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int64, Int64, Ref{Ptr{Cvoid}}),
		ctx.h, d, dims64, spacing, m, tp, n, sp, length(kinds32), kinds32, sills, ranges, rot, bet, first(rows) - 1, length(rows), out))
	op = KernelCrossCovMatrix(out[], n, ctx, rows)
	finalizer(freeop, op)
	return op
end

"LowRankCovMatrix(samples) -- src/lowrank.jl:14-30 (the mean is removed on the device)"
function LowRankCovMatrix(samples::Vector{Vector{Float64}}; ctx::Context=context())
	S = reduce(hcat, samples)
	buf = upload!(DeviceMatrix(ctx, GSI_LAYOUT_COLMAJOR, size(S)...), S)
	out = Ref{Ptr{Cvoid}}(C_NULL)
	check(ccall((:gsi_op_lowrankcov, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Ref{Ptr{Cvoid}}), ctx.h, buf.h, 1, out))
	op = LowRankCovMatrix(out[], buf, ctx, 1:size(S, 1))
	finalizer(freeop, op)
	return op
end

function Base.size(op::Operator)
	m = Ref{Int64}(0); n = Ref{Int64}(0)
	check(ccall((:gsi_op_size, LIB), Int32, (Ptr{Cvoid}, Ref{Int64}, Ref{Int64}), op.h, m, n))
	return (Int(m[]), Int(n[]))
end
Base.size(op::Operator, i::Int) = (i == 1 || i == 2) ? size(op)[i] : error("there is no $i-th dimension in a $(typeof(op))")
Base.eltype(::Operator) = Float64
Base.adjoint(op::Union{KernelCovMatrix, LowRankCovMatrix}) = op      # symmetric (src/lowrank.jl:38-44)
Base.transpose(op::Union{KernelCovMatrix, LowRankCovMatrix}) = op

"lazy adjoint of a non-symmetric operator (dense, cross-covariance), so that `A' * X` maps onto gsi_op_apply(trans = 1)"
struct AdjointOperator{T<:Operator}; parent::T; end
Base.adjoint(op::Union{DenseOperator, KernelCrossCovMatrix}) = AdjointOperator(op)
Base.adjoint(a::AdjointOperator) = a.parent
Base.size(a::AdjointOperator) = reverse(size(a.parent))
Base.size(a::AdjointOperator, i::Int) = size(a)[i]

"op(A) * X through the device: this worker's rows of the product (dense A'X: all rows, summed over workers)"
function apply(op::Operator, trans::Bool, X::Matrix{Float64})
	ctx = op.ctx
	t = (trans && !issym(op)) ? Int32(1) : Int32(0)
	outrows = t == 1 ? size(op, 2) : length(op.rows)
	Y = Matrix{Float64}(undef, outrows, size(X, 2))
	for c0 = 1:MAXCOLS:size(X, 2)                                   # passes of at most 256 columns
		cols = c0:min(c0 + MAXCOLS - 1, size(X, 2))
		Xd = upload!(DeviceMatrix(ctx, GSI_LAYOUT_TALL, size(X, 1), length(cols)), X[:, cols])
		Yd = DeviceMatrix(ctx, GSI_LAYOUT_TALL, outrows, length(cols))
		check(ccall((:gsi_op_apply, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{Cvoid}, Ptr{Cvoid}), op.h, t, Xd.h, Yd.h))
		Y[:, cols] = download(Yd)
	end
	return Y
end

Base.:*(op::Operator, X::Matrix{Float64}) = apply(op, false, X)                       # src/lowrank.jl:115-121
Base.:*(op::Operator, x::Vector{Float64}) = vec(apply(op, false, reshape(x, :, 1)))    # src/lowrank.jl:135-139
Base.:*(a::AdjointOperator, X::Matrix{Float64}) = apply(a.parent, true, X)            # A' * Q, RandMatFact.jl:67
Base.:*(a::AdjointOperator, x::Vector{Float64}) = vec(apply(a.parent, true, reshape(x, :, 1)))
# `B' * A = (A' * B)'` (src/lowrank.jl:131-133; RandMatFact.jl:85 `Q' * A`)
Base.:*(Bt::LinearAlgebra.Adjoint{Float64, Matrix{Float64}}, op::Operator) = Matrix(apply(op, true, Matrix(parent(Bt)))')

"""
covsolve(C, B; rtol=1e-10, maxiter=nothing, rank=0, seed=nothing, full=false) -> (X, info)

X = C \\ B for a square kernel-covariance operator (KernelCovMatrix, KernelCovGrid, KernelCovModel, KernelCovModelGrid;
nugget included) by gsi_kernelcov_solve: one preconditioned CG recurrence per column of B (k <= 1024), sharing one
operator product per iteration; column j stops at ||r_j|| <= rtol ||b_j||.  rank > 0 draws an n x rank Gaussian sketch
(`randn`, after `Random.seed!(seed)` when a seed is given) for the randomized Nystrom preconditioner (rank <= 256,
rank < n).  maxiter = nothing means n.  info: iterations, relres (true ||b - C x|| / ||b||), nystrom_eigenvalues.
Multi-GPU: this worker's rows of X unless full = true.
"""
function covsolve(C::KernelCovMatrix, B::VecOrMat{Float64}; rtol::Float64=1e-10, maxiter::Union{Nothing, Int}=nothing,
		rank::Int=0, seed::Union{Nothing, Int}=nothing, full::Bool=false)
	seed === nothing || Random.seed!(seed)
	n = size(C, 2)
	Bm = Matrix{Float64}(reshape(B, n, :))
	k = size(Bm, 2)
	Bd = upload!(DeviceMatrix(C.ctx, GSI_LAYOUT_TALL, n, k), Bm)
	Om = rank > 0 ? upload!(DeviceMatrix(C.ctx, GSI_LAYOUT_TALL, n, rank), randn(n, rank)) : nothing
	Xd = DeviceMatrix(C.ctx, GSI_LAYOUT_TALL, (full || C.ctx.world == 1) ? n : length(C.rows), k)
	iters = zeros(Int64, k); relres = zeros(k); lambda = zeros(max(rank, 1))
	status = GC.@preserve iters relres lambda ccall((:gsi_kernelcov_solve, LIB), Int32,
		(Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Float64, Int64, Ptr{Cvoid}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}),
		C.h, Bd.h, Om === nothing ? C_NULL : Om.h, rtol, maxiter === nothing ? n : maxiter, Xd.h, iters, relres, lambda)
	(status == 0 || status == 10) || check(status)
	X = download(Xd)
	X = B isa Vector ? vec(X) : X
	info = (iterations=iters, relres=relres, nystrom_eigenvalues=lambda[1:rank])
	status == 10 && throw(CovSolveNoConvergence(lasterror(), X, info))     # X, iterations and relres are filled
	return X, info
end

"a column of covsolve did not reach rtol within maxiter iterations; `X` and `info` are those of the returned solve"
struct CovSolveNoConvergence <: Exception
	msg::String
	X::VecOrMat{Float64}
	info::NamedTuple
end
Base.showerror(io::IO, e::CovSolveNoConvergence) = print(io, "CovSolveNoConvergence: ", e.msg)

"""
krige(kinds, sills, ranges, sources, y, targets; rotations, betas, nugget=0.0, drift=nothing, rtol=1e-10, rank=0,
      seed=nothing, method=:cg, variance=false) -> (yhat, beta, w) or (yhat, beta, w, var)

Dual-form kriging at the targets (d x m) from observations y at the sources (d x n) under the nested model of
KernelCovModel plus `nugget`: one solve of C [alpha | B_F] = [y | F], beta = (F' B_F) \\ (F' alpha),
w = alpha - B_F beta, yhat = F_T beta + C(T, S) w (multi-GPU: this worker's block of target rows, as `Cx * w`).  drift = nothing: simple kriging; :constant: ordinary kriging;
(F_sources n x p, F_targets m x p): universal kriging / kriging with external drift.  method = :cg solves by covsolve
(rtol, rank, seed apply); method = :cholesky by the dense factor covchol (one GPU, about 8 n^2 bytes), and
variance = true then appends the kriging variance of the noise-free value at every target (covchol_variance).
"""
function krige(kinds::Vector{<:Integer}, sills::Vector{Float64}, ranges::Matrix{Float64}, sources::Matrix{Float64},
		y::Vector{Float64}, targets::Matrix{Float64}; rotations::Union{Nothing, Array{Float64, 3}}=nothing,
		betas::Union{Nothing, Vector{Float64}}=nothing, nugget=0.0, drift=nothing, rtol::Float64=1e-10, rank::Int=0,
		seed::Union{Nothing, Int}=nothing, method::Symbol=:cg, variance::Bool=false)
	method in (:cg, :cholesky) || throw(ArgumentError("krige: method must be :cg or :cholesky"))
	variance && method === :cg && throw(ArgumentError("krige: variance = true needs method = :cholesky (on the CG " *
		"path the variance costs one iterative solve per target)"))
	n, m = size(sources, 2), size(targets, 2)
	F, FT = drift === nothing ? (zeros(n, 0), zeros(m, 0)) :
		drift === :constant ? (ones(n, 1), ones(m, 1)) : (Matrix{Float64}(drift[1]), Matrix{Float64}(drift[2]))
	C = KernelCovModel(kinds, sills, ranges, sources; rotations=rotations, betas=betas, nugget=nugget)
	Cx = KernelCrossCov(kinds, sills, ranges, targets, sources; rotations=rotations, betas=betas)
	fct = method === :cholesky ? covchol(C) : nothing
	X = fct === nothing ? covsolve(C, hcat(y, F); rtol=rtol, rank=rank, seed=seed, full=true)[1] : covchol_solve(fct, hcat(y, F))
	alpha, BF = X[:, 1], X[:, 2:end]
	beta = size(F, 2) > 0 ? (F' * BF) \ (F' * alpha) : zeros(0)
	w = alpha - BF * beta
	yhat = FT[Cx.rows, :] * beta + Cx * w                          # this worker's target rows (all on one GPU)
	variance || return yhat, beta, w
	return yhat, beta, w, covchol_variance(fct, Cx; drift=size(F, 2) > 0 ? (F, FT) : nothing)
end

"""
covchol(C; diag=nothing) -> CovCholesky

Dense Cholesky factor C + Diagonal(diag) = L L' of a square kernel-covariance operator (KernelCovMatrix, KernelCovGrid,
KernelCovModel, KernelCovModelGrid; nugget included) on the device by gsi_kernelcov_chol (gsi_kernelcov_chol_diag with a
per-point diagonal of n values): one GPU, about 8 n^2 bytes.  A non-positive pivot throws
LinearAlgebra.PosDefException(column).  Freed by its finalizer.
"""
mutable struct CovCholesky; h::Ptr{Cvoid}; n::Int; ctx::Context; end
function covchol(C::KernelCovMatrix; diag::Union{Nothing, Vector{Float64}}=nothing)
	out = Ref{Ptr{Cvoid}}(C_NULL)
	col = Ref{Int64}(0)
	if diag === nothing
		check(ccall((:gsi_kernelcov_chol, LIB), Int32, (Ptr{Cvoid}, Ptr{Ptr{Cvoid}}, Ptr{Int64}), C.h, out, col))
	else
		length(diag) == size(C, 2) || throw(DimensionMismatch("covchol: diag has $(length(diag)) values, C is $(size(C, 2)) x $(size(C, 2))"))
		check(ccall((:gsi_kernelcov_chol_diag, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Ptr{Cvoid}}, Ptr{Int64}),
			C.h, diag, out, col))
	end
	f = CovCholesky(out[], size(C, 2), C.ctx)
	finalizer(x->ccall((:gsi_chol_free, LIB), Int32, (Ptr{Cvoid},), x.h), f)    # idempotent, never throws
	return f
end

"log det C = 2 sum log L[i, i] (Gaussian log-likelihood of covariance parameters)"
function covchol_logdet(f::CovCholesky)
	v = Ref{Float64}(0.0)
	check(ccall((:gsi_chol_logdet, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}), f.h, v))
	return v[]
end

"C \\ B (half = false) or L \\ B (half = true), any number of columns (1024 per device call)"
function covchol_solve(f::CovCholesky, B::VecOrMat{Float64}; half::Bool=false)
	Bm = Matrix{Float64}(reshape(B, f.n, :))
	X = similar(Bm)
	for c0 in 1:1024:size(Bm, 2)
		cols = c0:min(c0 + 1023, size(Bm, 2))
		Bd = upload!(DeviceMatrix(f.ctx, GSI_LAYOUT_TALL, f.n, length(cols)), Bm[:, cols])
		check(ccall((:gsi_chol_solve, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{Cvoid}, Ptr{Cvoid}), f.h, Int32(half), Bd.h, Bd.h))
		X[:, cols] = download(Bd)
	end
	return B isa Vector ? vec(X) : X
end

"""
covchol_variance(f, Cx; drift=nothing) -> var (m)

Kriging variance of the noise-free value at the targets of Cx = KernelCrossCov(..., targets, sources) whose sources are
the factor's points: c(t, t) - ||L \\ c_t||^2 (drift = nothing), plus r' (G'G) \\ r, G = L \\ F_s, r = f_t - G' (L \\ c_t)
with drift = :constant or (F_sources n x p, F_targets m x p), p <= 32.
"""
function covchol_variance(f::CovCholesky, Cx::KernelCrossCovMatrix; drift=nothing)
	m = size(Cx, 1)
	F, FT = drift === nothing ? (zeros(f.n, 0), zeros(m, 0)) :
		drift === :constant ? (ones(f.n, 1), ones(m, 1)) : (Matrix{Float64}(drift[1]), Matrix{Float64}(drift[2]))
	p = size(F, 2)
	var = zeros(m)
	GC.@preserve F FT var check(ccall((:gsi_chol_krige_variance, LIB), Int32,
		(Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}),
		f.h, Cx.h, p > 0 ? pointer(F) : C_NULL, p > 0 ? pointer(FT) : C_NULL, p, var))
	return var
end

"""
covchol_simulate(f, Xi; ncond=0, y=nothing, drift=nothing) -> Z ((n - ncond) x k)

Realisations at the last n - ncond points of a factor of the joint matrix [sources; targets] (gsi_chol_simulate):
Z = F_t B + L(T, :) V from the standard normals Xi (n x k, any k; 1024 columns per device call), conditioned on y
(ncond values) at the first ncond points with drift = nothing (simple kriging), :constant or (F_sources, F_targets),
p <= 32.  Xi = 0 gives the kriging estimate; ncond = 0 gives unconditional samples L Xi.
"""
function covchol_simulate(f::CovCholesky, Xi::VecOrMat{Float64}; ncond::Int=0, y=nothing, drift=nothing)
	ns, m = ncond, f.n - ncond
	drift !== nothing && ns == 0 && throw(ArgumentError("covchol_simulate: a drift needs conditioning data (ncond > 0)"))
	F, FT = drift === nothing ? (zeros(ns, 0), zeros(m, 0)) :
		drift === :constant ? (ones(ns, 1), ones(m, 1)) : (Matrix{Float64}(drift[1]), Matrix{Float64}(drift[2]))
	p = size(F, 2)
	yv = y === nothing ? zeros(0) : Vector{Float64}(y)
	length(yv) == ns || throw(DimensionMismatch("covchol_simulate: y has $(length(yv)) values, ncond is $ns"))
	X = Matrix{Float64}(reshape(Xi, f.n, :))
	Z = zeros(m, size(X, 2))
	for c0 in 1:1024:size(X, 2)
		cols = c0:min(c0 + 1023, size(X, 2))
		Xd = upload!(DeviceMatrix(f.ctx, GSI_LAYOUT_TALL, f.n, length(cols)), X[:, cols])
		Zd = DeviceMatrix(f.ctx, GSI_LAYOUT_TALL, m, length(cols))
		GC.@preserve yv F FT check(ccall((:gsi_chol_simulate, LIB), Int32,
			(Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Cvoid}, Ptr{Cvoid}),
			f.h, ns, ns > 0 ? pointer(yv) : C_NULL, p > 0 ? pointer(F) : C_NULL, p > 0 ? pointer(FT) : C_NULL, p,
			Xd.h, Zd.h))
		Z[:, cols] = download(Zd)
	end
	return Z
end

"""
covloglik(C, y; drift=nothing, reml=false, grad=false) -> (value, beta) or (value, beta, gradient)

Gaussian log-likelihood of the observations y under the square kernel-covariance operator C (nugget included), the
drift coefficients profiled out by GLS (gsi_kernelcov_loglik; one dense factorisation on one GPU, about 8 n^2 bytes).
drift = nothing, :constant or an n x p matrix F (p <= 32).  reml = false: -1/2 (n log 2 pi + log det C + q); reml = true:
-1/2 ((n - p) log 2 pi + log det C + log det F'C^-1 F + q), without log det F'F; q the GLS residual quadratic form.  With
grad = true the exact gradient for, per structure, the sill then the d ranges, and last the nugget (not on grid
operators).  A non-positive pivot throws LinearAlgebra.PosDefException(column).
"""
function covloglik(C::KernelCovMatrix, y::Vector{Float64}; drift=nothing, reml::Bool=false, grad::Bool=false)
	n = size(C, 2)
	F = drift === nothing ? zeros(n, 0) : drift === :constant ? ones(n, 1) : Matrix{Float64}(drift)
	p = size(F, 2)
	val = Ref{Float64}(0.0)
	col = Ref{Int64}(0)
	beta = zeros(max(p, 1))
	g = zeros(C.nparams)
	GC.@preserve y F beta g check(ccall((:gsi_kernelcov_loglik, LIB), Int32,
		(Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}),
		C.h, y, p > 0 ? pointer(F) : C_NULL, p, Int32(reml), val, beta, grad ? pointer(g) : C_NULL, col))
	return grad ? (val[], beta[1:p], g) : (val[], beta[1:p])
end

"""
covchol_crossval(f, y; drift=nothing, groups=nothing) -> (prediction, error, variance, logpdf)

Leave-one-out (groups = nothing) or leave-group-out cross-validation of kriging on the factor (gsi_chol_crossval,
Dubrule 1983): for each group B (a vector of 1..128 distinct 1-based point indices) the prediction of y[B] from all
other points, the drift (nothing, :constant or an n x p matrix, p <= 32) re-estimated by GLS from them, its error
y[B] - prediction, the error variance of the observation (nugget included: the noise-free kriging variance is
variance - nugget) and the Gaussian log-density of y[B] given the other points.  prediction, error and variance have n
entries in point order, NaN at points not held out; logpdf one per group.  A group whose drift the other points cannot
identify throws LinearAlgebra.PosDefException(group).
"""
function covchol_crossval(f::CovCholesky, y::Vector{Float64}; drift=nothing, groups=nothing)
	n = f.n
	length(y) == n || throw(DimensionMismatch("covchol_crossval: y has $(length(y)) values, the factor is $n x $n"))
	F = drift === nothing ? zeros(n, 0) : drift === :constant ? ones(n, 1) : Matrix{Float64}(drift)
	p = size(F, 2)
	ng = groups === nothing ? n : length(groups)
	ptr = groups === nothing ? Int64[] : vcat(0, cumsum(Int64[length(g) for g in groups]))
	idx = groups === nothing ? Int64[] : Int64[i - 1 for g in groups for i in g]
	m = groups === nothing ? n : Int(ptr[end])
	err, var, lpd = zeros(max(m, 1)), zeros(max(m, 1)), zeros(max(ng, 1))
	failed = Ref{Int64}(0)
	status = GC.@preserve y F ptr idx err var lpd ccall((:gsi_chol_crossval, LIB), Int32,
		(Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64},
		 Ptr{Float64}, Ptr{Int64}),
		f.h, y, p > 0 ? pointer(F) : C_NULL, p, ng, groups === nothing ? C_NULL : pointer(ptr),
		groups === nothing ? C_NULL : pointer(idx), err, var, lpd, failed)
	failed[] > 0 && throw(LinearAlgebra.PosDefException(Int(failed[])))
	check(status)
	pts = groups === nothing ? collect(1:n) : idx .+ 1
	e, v = fill(NaN, n), fill(NaN, n)
	e[pts] = err[1:m]
	v[pts] = var[1:m]
	pred = y .- e
	return pred, e, v, lpd[1:ng]
end

"""
simulate(kinds, sills, ranges, targets, nreal; rotations, betas, sources=nothing, y=nothing, nugget=0.0,
         target_nugget=0.0, drift=nothing, seed=nothing) -> Z (m x nreal)

Gaussian realisations at the targets (d x m) under the nested model of KernelCovModel, conditioned on y at the sources
(observation noise `nugget`) or unconditional (sources = nothing): LU simulation on one dense factor of the joint matrix
of [sources targets] plus Diagonal(nugget at the sources, target_nugget at the targets) (covchol, covchol_simulate; one
GPU, about 8 (ns + m)^2 bytes).  The standard normals are drawn on the host by `randn` (after `Random.seed!(seed)` when
a seed is given).  drift as in krige, conditional simulation only.
"""
function simulate(kinds::Vector{<:Integer}, sills::Vector{Float64}, ranges::Matrix{Float64}, targets::Matrix{Float64},
		nreal::Int; rotations::Union{Nothing, Array{Float64, 3}}=nothing, betas::Union{Nothing, Vector{Float64}}=nothing,
		sources::Union{Nothing, Matrix{Float64}}=nothing, y=nothing, nugget=0.0, target_nugget=0.0, drift=nothing,
		seed::Union{Nothing, Int}=nothing)
	sources === nothing && drift !== nothing && throw(ArgumentError("simulate: a drift needs conditioning data"))
	S = sources === nothing ? zeros(size(targets, 1), 0) : sources
	ns, m = size(S, 2), size(targets, 2)
	seed === nothing || Random.seed!(seed)
	Xi = randn(ns + m, nreal)
	C = KernelCovModel(kinds, sills, ranges, hcat(S, targets); rotations=rotations, betas=betas, nugget=0.0)
	f = covchol(C; diag=vcat(fill(Float64(nugget), ns), fill(Float64(target_nugget), m)))
	return covchol_simulate(f, Xi; ncond=ns, y=ns > 0 ? y : nothing, drift=drift)
end

module RandMatFact
import ..GeostatInversionB200: LIB, check, context, Operator, DenseOperator, DeviceMatrix, upload!, download,
	GSI_LAYOUT_TALL, GSI_NORMALISER_LU_REF, issym
import LinearAlgebra

asoperator(A::Operator) = A
asoperator(A::Matrix{Float64}) = DenseOperator(A)

"randsvd(A, K, p, q) -- reference src/RandMatFact.jl:83-90 (Omega drawn on the host, :54).  On a multi-worker context every worker draws the same Omega (seed identically) and receives its own rows of Z; pass `full=true` for all rows."
function randsvd(A, K::Int, p::Int, q::Int; full::Bool=false)
	q < 0 && error("parameter numiterations should be positive, but numiterations=$q")
	op = asoperator(A)
	n = size(op, 2)
	Omega = randn(n, K + p)                              # same host RNG stream as the reference
	Om = upload!(DeviceMatrix(op.ctx, GSI_LAYOUT_TALL, n, K + p), Omega)
	zrows = (full || !issym(op)) ? n : length(op.rows)
	Z = DeviceMatrix(op.ctx, GSI_LAYOUT_TALL, zrows, K + p)
	check(ccall((:gsi_randsvd, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int64, Int64, Int32, Ptr{Cvoid}, Ptr{Float64}),
		op.h, Om.h, K, p, q, GSI_NORMALISER_LU_REF, Z.h, C_NULL))
	return download(Z)
end

"rangefinder(A, l, numiterations) -- reference src/RandMatFact.jl:50-80"
function rangefinder(A, l::Int64, numiterations::Int64)
	numiterations < 0 && error("parameter numiterations should be positive, but numiterations=$numiterations")
	op = asoperator(A)
	n = size(op, 2)
	Om = upload!(DeviceMatrix(op.ctx, GSI_LAYOUT_TALL, n, l), randn(n, l))
	Q = DeviceMatrix(op.ctx, GSI_LAYOUT_TALL, length(op.rows), l)
	check(ccall((:gsi_rangefinder_fixed, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int32, Ptr{Cvoid}), op.h, Om.h, numiterations, GSI_NORMALISER_LU_REF, Q.h))
	return download(Q)
end

"""
rangefinder(A; epsilon=1e-8, r=10) -- reference src/RandMatFact.jl:15-48 (HMT algorithm 4.2).
The r start vectors (`randn(n, r)`, :20) and the vectors the reference draws one by one with
`randn!(omega)` (:36) are drawn here in the same order and handed to the library in blocks of
one matrix, so a run consumes the same random stream as the reference up to the point where it
stops (the reference draws nothing after convergence; this shim draws
the whole set of min(m, n) vectors up front).
"""
function rangefinder(A; epsilon::Float64=1e-8, r::Int=10, block::Union{Nothing, Int}=nothing)
	op = asoperator(A)
	m, n = size(op)
	if block !== nothing                                 # OPT-IN blocked finder (not the parity mode): one GEMM pass over A per block
		maxvec = min(m, n)
		oms = upload!(DeviceMatrix(op.ctx, GSI_LAYOUT_COLMAJOR, n, maxvec), randn(n, maxvec))
		Q = DeviceMatrix(op.ctx, GSI_LAYOUT_COLMAJOR, m, maxvec)
		j = Ref{Int64}(0)
		check(ccall((:gsi_rangefinder_adaptive_blocked, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Float64, Int64, Ptr{Cvoid}, Ref{Int64}),
			op.h, oms.h, epsilon, block, Q.h, j))
		return download(Q)[:, 1:j[]]
	end
	Om0 = upload!(DeviceMatrix(op.ctx, GSI_LAYOUT_TALL, n, r), randn(n, r))
	maxvec = min(m, n)
	oms = upload!(DeviceMatrix(op.ctx, GSI_LAYOUT_COLMAJOR, n, maxvec), randn(n, maxvec))
	Q = DeviceMatrix(op.ctx, GSI_LAYOUT_COLMAJOR, m, maxvec)
	j = Ref{Int64}(0)
	check(ccall((:gsi_rangefinder_adaptive, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Float64, Int64, Ptr{Cvoid}, Ref{Int64}),
		op.h, Om0.h, oms.h, epsilon, r, Q.h, j))
	return download(Q)[:, 1:j[]]
end

"eig_nystrom(A, Q) -> (U, Sigmavec) -- reference src/RandMatFact.jl:92-102"
function eig_nystrom(A, Q::Matrix{Float64})
	op = asoperator(A)
	l = size(Q, 2)
	Qd = upload!(DeviceMatrix(op.ctx, GSI_LAYOUT_TALL, size(Q)...), Q)
	U = DeviceMatrix(op.ctx, GSI_LAYOUT_TALL, size(op, 1), l)
	Sigmavec = Vector{Float64}(undef, l)
	GC.@preserve Sigmavec check(ccall((:gsi_eig_nystrom, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}), op.h, Qd.h, U.h, Sigmavec))
	return download(U), Sigmavec
end
end # RandMatFact

"""
FFTRF.powerlaw_structuredgrid (src/FFTRF.jl:83-100) on the device, for a batch of fields: the phases
`randn(size(S))` (:75) are drawn here, per field, in the reference's order; the fields stay on the
device as the columns of an n x numfields matrix (gsi_fftrf_powerlaw).
"""
module FFTRF
import ..GeostatInversionB200: LIB, check, context, Context, DeviceMatrix, upload!, download, GSI_LAYOUT_COLMAJOR

doubledsize(Ns::Vector{Int}) = length(Ns) == 2 ? (2 * Ns[2], 2 * Ns[1]) : (2 * Ns[2], 2 * Ns[1], 2 * Ns[3])   # size(S), :45,52

function samplefieldsdevice(Ns::Vector{Int}, k0::Number, dk::Number, beta::Number, numfields::Int; ctx::Context=context())
	(length(Ns) == 2 || length(Ns) == 3) || error("unsupported dimension: $(length(Ns))")
	big = prod(doubledsize(Ns))
	phi = Matrix{Float64}(undef, big, numfields)
	for f = 1:numfields
		phi[:, f] = vec(randn(doubledsize(Ns)))              # mulbyphi, :74-75
	end
	phid = upload!(DeviceMatrix(ctx, GSI_LAYOUT_COLMAJOR, big, numfields), phi)
	out = DeviceMatrix(ctx, GSI_LAYOUT_COLMAJOR, prod(Ns), numfields)
	Ns64 = Int64.(Ns)
	GC.@preserve Ns64 check(ccall((:gsi_fftrf_powerlaw, LIB), Int32,
		(Ptr{Cvoid}, Int32, Ptr{Int64}, Float64, Float64, Float64, Ptr{Cvoid}, Ptr{Cvoid}),
		ctx.h, length(Ns), Ns64, k0, dk, beta, phid.h, out.h))
	return out
end

"powerlaw_structuredgrid(Ns, k0, dk, beta) -> Array of size Ns (src/FFTRF.jl:83-100)"
powerlaw_structuredgrid(Ns::Vector, k0::Number, dk::Number, beta::Number) =
	reshape(download(samplefieldsdevice(Vector{Int}(Ns), k0, dk, beta, 1))[:, 1], Ns...)

"a `samplefield` that getxis recognises and evaluates as ONE batch on the device"
struct PowerLawSampler
	Ns::Vector{Int}
	k0::Float64
	dk::Float64
	beta::Float64
end
(s::PowerLawSampler)() = vec(powerlaw_structuredgrid(s.Ns, s.k0, s.dk, s.beta))
end # FFTRF

function randsvdwithseed(Q, numxis, p, q, seed::Nothing)
	return RandMatFact.randsvd(Q, numxis, p, q)
end
function randsvdwithseed(Q, numxis, p, q, seed::Int)
	Random.seed!(seed)                                   # src/GeostatInversion.jl:24-27
	return RandMatFact.randsvd(Q, numxis, p, q)
end

"getxis(Q, numxis, p, q=3, seed=nothing) -- src/GeostatInversion.jl:63-70; Q::Matrix or any Operator"
function getxis(Q::Union{Matrix{Float64}, Operator}, numxis::Int, p::Int, q::Int=3, seed=nothing)
	Z = randsvdwithseed(Q, numxis, p, q, seed)
	return [Z[:, i] for i = 1:numxis]
end

"getxis(Val{:iwantfields}, samplefield, numfields, numxis, p, q=3, seed=nothing) -> (xis, fields) -- src/GeostatInversion.jl:29-38"
function getxis(::Type{Val{:iwantfields}}, samplefield::Function, numfields::Int, numxis::Int, p::Int, q::Int=3, seed=nothing)
	fields = Distributed.pmap(i->samplefield(), 1:numfields; batch_size=ceil(Int, numfields / max(1, Distributed.nworkers())))
	lrcm = LowRankCovMatrix(Vector{Vector{Float64}}(fields))
	Z = randsvdwithseed(lrcm, numxis, p, q, seed)
	xis = Array{Array{Float64, 1}}(undef, numxis)
	for i = 1:numxis
		xis[i] = Z[:, i]
	end
	return xis, fields
end

"getxis for the device sampler: fields generated, mean-removed and factored without leaving the device"
function getxis(::Type{Val{:iwantfields}}, sampler::FFTRF.PowerLawSampler, numfields::Int, numxis::Int, p::Int, q::Int=3, seed=nothing)
	ctx = context()
	Sd = FFTRF.samplefieldsdevice(sampler.Ns, sampler.k0, sampler.dk, sampler.beta, numfields; ctx=ctx)
	S = download(Sd)                                     # the raw fields the reference also returns (before mean removal)
	out = Ref{Ptr{Cvoid}}(C_NULL)
	check(ccall((:gsi_op_lowrankcov, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Ref{Ptr{Cvoid}}), ctx.h, Sd.h, 1, out))
	lrcm = LowRankCovMatrix(out[], Sd, ctx, 1:Sd.rows)
	finalizer(freeop, lrcm)
	Z = randsvdwithseed(lrcm, numxis, p, q, seed)
	return [Z[:, i] for i = 1:numxis], [S[:, i] for i = 1:numfields]
end
getxis(sampler::FFTRF.PowerLawSampler, numfields::Int, numxis::Int, p::Int, q::Int=3, seed=nothing) =
	getxis(Val{:iwantfields}, sampler, numfields, numxis, p, q, seed)[1]

"getxis(samplefield, numfields, numxis, p, q=3, seed=nothing) -- src/GeostatInversion.jl:58-61"
function getxis(samplefield::Function, numfields::Int, numxis::Int, p::Int, q::Int=3, seed=nothing)
	xis, _ = getxis(Val{:iwantfields}, samplefield, numfields, numxis, p, q, seed)
	return xis
end

# ---------------------------------------------------------------------------------------------
# PCGA / RGA drivers behind the reference's keyword surface (src/lsqr.jl:20-63,
# src/direct.jl:21-67, src/GeostatInversion.jl:101-105).  Transcription of the tested Python
# host geostatinversion.jl_b200/pcga.py.  The user's forward model stays a Julia function run
# under `pmap`, exactly as in the reference; the batch of K+3 parameter vectors, the
# saddle-point solve and the update run on the device.

splitR(R::Number, nobs) = (fill(Float64(R), nobs), nothing)
splitR(R::AbstractVector, nobs) = (Vector{Float64}(R), nothing)
splitR(R::LinearAlgebra.Diagonal, nobs) = (Vector{Float64}(R.diag), nothing)
function splitR(R::SparseArrays.SparseMatrixCSC, nobs)
	d = Vector{Float64}(LinearAlgebra.diag(R))
	return SparseArrays.nnz(SparseArrays.dropzeros(R - SparseArrays.spdiagm(0=>d))) == 0 ? (d, nothing) : (nothing, Matrix{Float64}(R))
end
splitR(R::AbstractMatrix, nobs) = (nothing, Matrix{Float64}(R))

function xistodevice(ctx::Context, xis::Vector{Vector{Float64}})
	length(xis) + 3 <= MAXWIDECOLS || throw(ArgumentError("at most $(MAXWIDECOLS - 3) xis (the batch of K+3 parameter vectors is one device iterate of at most 1024 columns)"))
	Zk = reduce(hcat, xis)
	return upload!(DeviceMatrix(ctx, GSI_LAYOUT_TALL, size(Zk)...), Zk)
end

"`paramstorun` batch (src/lsqr.jl:37-43 == src/direct.jl:39-45) as the columns of an n x (K+3) matrix"
function paramstorun(ctx::Context, Zk::DeviceMatrix, K::Int, s::Vector{Float64}, X::Vector{Float64}, delta::Float64)
	P = DeviceMatrix(ctx, GSI_LAYOUT_TALL, Zk.rows, K + 3)
	GC.@preserve s X check(ccall((:gsi_pcga_paramstorun, LIB), Int32,
		(Ptr{Cvoid}, Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Float64, Ptr{Cvoid}), ctx.h, Zk.h, K, s, X, delta, P.h))
	return download(P)
end

# x = lsqr(PCGALowRankMatrix(etas, HX, R), b) (src/lsqr.jl:53-54) or pinv(bigA) * b (src/direct.jl:49-58)
function saddlesolve(ctx::Context, E::Matrix{Float64}, HX::Vector{Float64}, R, b::Vector{Float64}, direct::Bool)
	nobs, K = size(E)
	rd, rD = splitR(R, nobs)
	rdp = rd === nothing ? Ptr{Float64}(C_NULL) : pointer(rd)
	rDp = rD === nothing ? Ptr{Float64}(C_NULL) : pointer(rD)
	x = Vector{Float64}(undef, nobs + 1)
	GC.@preserve E HX rd rD b x begin
		if direct
			check(ccall((:gsi_pcga_direct_solve, LIB), Int32,
				(Ptr{Cvoid}, Int64, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}),
				ctx.h, nobs, K, E, nobs, HX, rdp, rDp, nobs, b, x, C_NULL))
		else
			check(ccall((:gsi_pcga_lsqr_solve, LIB), Int32,
				(Ptr{Cvoid}, Int64, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Float64, Float64, Float64, Int64, Ptr{Float64}, Ptr{Int64}, Ptr{Int32}),
				ctx.h, nobs, K, E, nobs, HX, rdp, rDp, nobs, b, 0.0, 0.0, 0.0, 0, x, C_NULL, C_NULL))
		end
	end
	return x
end

"""
The `PCGALowRankMatrix` of src/lowrank.jl:32-36 with its `mul!` on the device (:83-97):
`[HQH' + R, HX; HX', 0]`, `HQH' = sum_i eta_i eta_i'`.  Method set of the reference type
(`size`, `eltype`, `adjoint`, `*`, `mul!`), so it can also be handed to a Julia-side solver.
"""
struct PCGALowRankMatrix
	E::Matrix{Float64}
	HX::Vector{Float64}
	R
	ctx::Context
end
PCGALowRankMatrix(etas::Vector{Vector{Float64}}, HX::Vector{Float64}, R; ctx::Context=context()) = PCGALowRankMatrix(reduce(hcat, etas), HX, R, ctx)
Base.size(A::PCGALowRankMatrix) = (length(A.HX) + 1, length(A.HX) + 1)
Base.size(A::PCGALowRankMatrix, i::Int) = (i == 1 || i == 2) ? length(A.HX) + 1 : error("there is no $i-th dimension in a PCGALowRankMatrix")
Base.eltype(::PCGALowRankMatrix) = Float64
Base.adjoint(A::PCGALowRankMatrix) = A
function LinearAlgebra.mul!(v::Vector{Float64}, A::PCGALowRankMatrix, x::Vector{Float64})
	nobs, K = size(A.E)
	rd, rD = splitR(A.R, nobs)
	rdp = rd === nothing ? Ptr{Float64}(C_NULL) : pointer(rd)
	rDp = rD === nothing ? Ptr{Float64}(C_NULL) : pointer(rD)
	GC.@preserve A rd rD x v check(ccall((:gsi_pcga_lowrank_matvec, LIB), Int32,
		(Ptr{Cvoid}, Int64, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}),
		A.ctx.h, nobs, K, A.E, nobs, A.HX, rdp, rDp, nobs, x, v))
	return v
end
Base.:*(A::PCGALowRankMatrix, x::Vector{Float64}) = LinearAlgebra.mul!(Vector{Float64}(undef, length(x)), A, x)

function pcgaiteration(forwardmodel::Function, s::Vector{Float64}, X::Vector{Float64}, Zk::DeviceMatrix, K::Int, R, y::Vector{Float64},
		delta::Float64, callback::Function, direct::Bool, ctx::Context)
	P = paramstorun(ctx, Zk, K, s, X, delta)
	results = Distributed.pmap(forwardmodel, [P[:, i] for i = 1:K + 3])          # src/lsqr.jl:44
	hs = results[K + 3]
	callback(s, hs)                                                             # src/direct.jl:47
	E = Matrix{Float64}(undef, length(hs), K)
	for i = 1:K
		E[:, i] = (results[i] - hs) / delta                                     # etas, :46-49
	end
	HX = (results[K + 1] - hs) / delta                                          # :50
	Hs = (results[K + 2] - hs) / delta                                          # :51
	b = [y - hs + Hs; 0.0]                                                      # :52
	x = saddlesolve(ctx, E, HX, R, b, direct)
	snew = Vector{Float64}(undef, Zk.rows)
	GC.@preserve X E x snew check(ccall((:gsi_pcga_update, LIB), Int32,
		(Ptr{Cvoid}, Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Int64, Int64, Ptr{Float64}, Ptr{Float64}),
		ctx.h, Zk.h, K, X, E, size(E, 1), size(E, 1), x, snew))                 # s = X*beta + sum xi_i (eta_i . xi_bar), :55-61
	return snew
end

function pcgaouter(forwardmodel, s0, X, xis, R, y, maxiters, delta, xtol, callback, direct, ctx)
	Zk = xistodevice(ctx, xis)
	K = length(xis)
	converged = false
	s = Vector{Float64}(s0)
	itercount = 0
	while !converged && itercount < maxiters                                    # src/lsqr.jl:24-31
		olds = s
		s = pcgaiteration(forwardmodel, s, Vector{Float64}(X), Zk, K, R, Vector{Float64}(y), Float64(delta), callback, direct, ctx)
		if LinearAlgebra.norm(s - olds) < xtol
			converged = true
		end
		itercount += 1
	end
	return s
end

# The library context is NOT part of the reference's keyword surface: the drivers below use the
# module's default context (`setcontext!`), so that `rga` can call ANY `pcgafunc` with exactly the
# keywords the reference forwards (maxiters, delta, xtol, callback; src/GeostatInversion.jl:102).

"pcgalsqr(forwardmodel, s0, X, xis, R, y; maxiters=5, delta=sqrt(eps(Float64)), xtol=1e-6) -- src/lsqr.jl:20-33 (+ callback, SURVEY F5)"
pcgalsqr(forwardmodel::Function, s0::Vector, X::Vector, xis::Array{Array{Float64, 1}, 1}, R, y::Vector;
		maxiters::Int=5, delta::Float64=sqrt(eps(Float64)), xtol::Float64=1e-6, callback=(s, obs_cal)->nothing) =
	pcgaouter(forwardmodel, s0, X, xis, R, y, maxiters, delta, xtol, callback, false, context())

"pcgadirect(forwardmodel, s0, X, xis, R, y; maxiters=5, delta=sqrt(eps(Float64)), xtol=1e-6, callback=(s, obs_cal)->nothing) -- src/direct.jl:21-35"
pcgadirect(forwardmodel::Function, s0::Vector, X::Vector, xis::Array{Array{Float64, 1}, 1}, R, y::Vector;
		maxiters::Int=5, delta::Float64=sqrt(eps(Float64)), xtol::Float64=1e-6, callback=(s, obs_cal)->nothing) =
	pcgaouter(forwardmodel, s0, X, xis, R, y, maxiters, delta, xtol, callback, true, context())

const pcga = pcgadirect                                                         # src/GeostatInversion.jl:105

"rga(forwardmodel, s0, X, xis, R, y, S; maxiters, delta, xtol, pcgafunc=pcgadirect, callback) -- src/GeostatInversion.jl:101-103"
function rga(forwardmodel::Function, s0::Vector, X::Vector, xis::Array{Array{Float64, 1}, 1}, R, y::Vector, S::Matrix{Float64};
		maxiters::Int=5, delta::Float64=sqrt(eps(Float64)), xtol::Float64=1e-6, pcgafunc=pcgadirect, callback=(s, obs_cal)->nothing)
	ctx = context()
	Nred, nobs = size(S)
	Sd = upload!(DeviceMatrix(ctx, GSI_LAYOUT_COLMAJOR, Nred, nobs), S)
	function sketch(V::Matrix{Float64})                                         # S * V on the tensor-core GEMM
		Vd = upload!(DeviceMatrix(ctx, GSI_LAYOUT_TALL, size(V)...), V)
		out = DeviceMatrix(ctx, GSI_LAYOUT_TALL, Nred, size(V, 2))
		check(ccall((:gsi_sketch_apply, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}), ctx.h, Sd.h, Vd.h, out.h))
		return download(out)
	end
	rd, rD = splitR(R, nobs)
	if rd === nothing
		SRS = reduce(hcat, [sketch(Matrix((rD * S')[:, c0:min(c0 + MAXCOLS - 1, Nred)])) for c0 = 1:MAXCOLS:Nred])   # dense R: S * (R * S')
	else
		SRS = Matrix{Float64}(undef, Nred, Nred)
		GC.@preserve rd SRS check(ccall((:gsi_sketch_cov, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64),
			ctx.h, Sd.h, rd, SRS, Nred))
	end
	# exactly the reference's call: x->S*forwardmodel(x), S*R*S', S*y and the four keywords (user-supplied pcgafunc welcome)
	return pcgafunc(x->vec(sketch(reshape(forwardmodel(x), :, 1))), s0, X, xis, SRS, vec(sketch(reshape(Vector{Float64}(y), :, 1)));
		maxiters=maxiters, delta=delta, xtol=xtol, callback=callback)
end

end
