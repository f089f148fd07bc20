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
mutable struct KernelCovMatrix <: Operator; h::Ptr{Cvoid}; n::Int; ctx::Context; rows::UnitRange{Int}; end
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
	op = KernelCovMatrix(out[], n, ctx, rows)
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
	op = KernelCovMatrix(out[], n, ctx, rows)
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
	op = KernelCovMatrix(out[], n, ctx, rows)
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
	op = KernelCovMatrix(out[], n, ctx, rows)
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
