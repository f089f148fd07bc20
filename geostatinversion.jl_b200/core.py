"""Host-side objects over the C ABI: context, device matrices, and the operator
types that play the role of the reference's duck-typed `A`
(size / A*Matrix / A' / Adjoint*A; reference src/RandMatFact.jl:52-55,67,70,85 and
the LowRankCovMatrix method set, src/lowrank.jl:38-60,115-133).
"""
import ctypes as C
import numpy as np

from . import _lib
from ._lib import (LAYOUT_TALL, LAYOUT_COLMAJOR, KERNEL_EXPONENTIAL, KERNEL_GAUSSIAN, KERNEL_POWERLAW,
                   KERNEL_MATERN32, KERNEL_MATERN52, KERNEL_SPHERICAL, MODEL_MAX_STRUCTURES, NORMALISER_LU_REF,
                   NORMALISER_QR, check)

_KINDS = {"exponential": KERNEL_EXPONENTIAL, "gaussian": KERNEL_GAUSSIAN, "powerlaw": KERNEL_POWERLAW,
          "matern32": KERNEL_MATERN32, "matern52": KERNEL_MATERN52, "spherical": KERNEL_SPHERICAL,
          KERNEL_EXPONENTIAL: KERNEL_EXPONENTIAL, KERNEL_GAUSSIAN: KERNEL_GAUSSIAN,
          KERNEL_POWERLAW: KERNEL_POWERLAW, KERNEL_MATERN32: KERNEL_MATERN32,
          KERNEL_MATERN52: KERNEL_MATERN52, KERNEL_SPHERICAL: KERNEL_SPHERICAL}


def _f64_colmajor(a):
    a = np.asarray(a, dtype=np.float64)
    if a.ndim == 1:
        a = a.reshape(-1, 1)
    if not a.flags.f_contiguous:
        a = np.asfortranarray(a)
    return a


def _pd(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


class Context:
    """One context per process and GPU (gsi_ctx_create).  No CPU fallback: raises
    NoDeviceError when no sm_100 device is visible."""

    def __init__(self, device=0, rank=0, world=1, unique_id=None):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        uid = None
        if world > 1:
            if unique_id is None or len(unique_id) != 128:
                raise ValueError("world > 1 needs the 128-byte NCCL unique id from rank 0")
            uid = C.create_string_buffer(bytes(unique_id), 128)
        check(self._lib.gsi_ctx_create(device, rank, world, uid, C.byref(self._h)))
        self.device, self.rank, self.world = device, rank, world

    @staticmethod
    def unique_id():
        buf = C.create_string_buffer(128)
        check(_lib.load().gsi_comm_unique_id(buf))
        return buf.raw

    def sync(self):
        check(self._lib.gsi_ctx_sync(self._h))

    def stream(self):
        s = C.c_void_p()
        check(self._lib.gsi_ctx_stream(self._h, C.byref(s)))
        return s.value or 0

    def launch_count(self, reset=False):
        n = C.c_int64()
        check(self._lib.gsi_ctx_launch_count(self._h, C.byref(n), 1 if reset else 0))
        return n.value

    def gemm_timing(self, enable=None):
        """Returns (ms, launches, flops) accumulated so far; enable=True/False (re)starts/stops."""
        ms, n, fl = C.c_double(), C.c_int64(), C.c_double()
        flag = -1 if enable is None else (1 if enable else 0)
        check(self._lib.gsi_ctx_gemm_timing(self._h, flag, C.byref(ms), C.byref(n), C.byref(fl)))
        return ms.value, n.value, fl.value

    def phase_timing(self, reset=False):
        """ms per phase recorded while gemm timing is on: products, lu, qr, small svd, back-multiply."""
        out = (C.c_double * 8)()
        check(self._lib.gsi_ctx_phase_timing(self._h, out, 1 if reset else 0))
        names = ["products", "lu", "qr", "svd_small", "backmul"]
        return {n: out[i] for i, n in enumerate(names)}

    def set_option(self, name, value):
        """Tuning knob (gsi_ctx_set_option), e.g. ("kcov.window", 8)."""
        check(self._lib.gsi_ctx_set_option(self._h, name.encode(), int(value)))

    def get_option(self, name):
        v = C.c_int64()
        check(self._lib.gsi_ctx_get_option(self._h, name.encode(), C.byref(v)))
        return v.value

    def pinned_empty(self, shape):
        """Column-major Float64 array in page-locked host memory (gsi_host_alloc): uploads from it are
        plain DMA.  The memory is released when the array (and every view of it) is gone."""
        shape = tuple(int(x) for x in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        count = int(np.prod(shape)) if shape else 1
        ptr = C.c_void_p()
        check(self._lib.gsi_host_alloc(self._h, max(count, 1) * 8, C.byref(ptr)))
        owner = _PinnedBlock(self, ptr)
        buf = (C.c_double * max(count, 1)).from_address(ptr.value)
        buf._gsi_owner = owner                     # the ctypes array keeps the block alive; NumPy keeps the ctypes array
        return np.frombuffer(buf, dtype=np.float64, count=count).reshape(shape, order="F")

    def close(self):
        if getattr(self, "_h", None) and self._h:
            self._lib.gsi_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _PinnedBlock:
    def __init__(self, ctx, ptr):
        self.ctx, self.ptr = ctx, ptr

    def __del__(self):
        try:
            if self.ptr:
                self.ctx._lib.gsi_host_free(self.ctx._h if self.ctx._h else None, self.ptr)
        except Exception:
            pass
        self.ptr = None


_default_ctx = None


def default_context():
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0, 0, 1)
    return _default_ctx


def set_default_context(ctx):
    global _default_ctx
    _default_ctx = ctx


class DeviceMatrix:
    """Opaque device buffer handle (gsi_buf): rows x cols Float64."""

    def __init__(self, ctx, rows, cols, layout=LAYOUT_TALL):
        self.ctx = ctx
        self._lib = ctx._lib
        self._h = C.c_void_p()
        check(self._lib.gsi_buf_alloc(ctx._h, layout, rows, cols, C.byref(self._h)))
        self.shape = (int(rows), int(cols))
        self.layout = layout

    @classmethod
    def from_host(cls, ctx, a, layout=LAYOUT_TALL):
        a = _f64_colmajor(a)
        m = cls(ctx, a.shape[0], a.shape[1], layout)
        m.upload(a)
        return m

    def upload(self, a):
        a = _f64_colmajor(a)
        if a.shape != self.shape:
            raise _lib.DimensionMismatch(_lib.ERR_DIMENSION_MISMATCH, f"upload: host {a.shape} vs device {self.shape}")
        check(self._lib.gsi_buf_upload(self._h, _pd(a), max(1, a.shape[0])))
        return self

    def upload_rows(self, row0, a):
        a = _f64_colmajor(a)
        check(self._lib.gsi_buf_upload_rows(self._h, row0, a.shape[0], _pd(a), max(1, a.shape[0])))
        return self

    def numpy(self, out=None):
        if out is None:
            out = np.empty(self.shape, dtype=np.float64, order="F")
        assert out.flags.f_contiguous and out.shape == self.shape and out.dtype == np.float64
        check(self._lib.gsi_buf_download(self._h, _pd(out), max(1, self.shape[0])))
        return out

    def rows_numpy(self, row0, nrows):
        out = np.empty((nrows, self.shape[1]), dtype=np.float64, order="F")
        check(self._lib.gsi_buf_download_rows(self._h, row0, nrows, _pd(out), max(1, nrows)))
        return out

    def zero(self):
        check(self._lib.gsi_buf_zero(self._h))

    def free(self):
        if getattr(self, "_h", None) and self._h:
            self._lib.gsi_buf_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _as_tall(ctx, X):
    if isinstance(X, DeviceMatrix):
        return X, False
    return DeviceMatrix.from_host(ctx, X, LAYOUT_TALL), True


class _Operator:
    """Common behaviour of the operator types (the reference's duck-typed `A`)."""
    symmetric = False

    def __init__(self, ctx):
        self.ctx = ctx
        self._lib = ctx._lib
        self._h = C.c_void_p()
        self._trans = False

    # size(A), size(A, i)  (1-based i like the reference, src/lowrank.jl:54-60)
    @property
    def shape(self):
        m, n = C.c_int64(), C.c_int64()
        check(self._lib.gsi_op_size(self._h, C.byref(m), C.byref(n)))
        return (n.value, m.value) if self._trans else (m.value, n.value)

    def size(self, i=None):
        if i is None:
            return self.shape
        if i in (1, 2):
            return self.shape[i - 1]
        raise ValueError(f"there is no {i}-th dimension in a {type(self).__name__}")

    @property
    def T(self):
        if self.symmetric:
            return self                                   # adjoint(A) = A, src/lowrank.jl:38-44
        return _TransposedView(self)

    adjoint = T

    def local_rows(self):
        return self.row0, self.mloc

    def apply(self, X, trans=False):
        """A*X (or A'*X).  X: ndarray or TALL DeviceMatrix holding all operand rows.
        Returns the same kind of object; on a sharded operator only this rank's rows
        (dense trans: all rows).  Host matrices wider than 256 columns are processed in
        256-column passes (a TALL device iterate holds at most 256 columns)."""
        if not isinstance(X, DeviceMatrix):
            Xh = np.asarray(X, dtype=np.float64)
            if Xh.ndim == 2 and Xh.shape[1] > 256:
                return np.concatenate([self.apply(Xh[:, c:c + 256], trans) for c in range(0, Xh.shape[1], 256)],
                                      axis=1)
        Xd, tmp = _as_tall(self.ctx, X)
        m, n = (self.shape if not self._trans else self.shape[::-1])
        sym = self.symmetric
        if sym or not trans:
            out_rows = self.mloc
        else:
            out_rows = n
        Y = DeviceMatrix(self.ctx, out_rows, Xd.shape[1], LAYOUT_TALL)
        check(self._lib.gsi_op_apply(self._h, 1 if (trans and not sym) else 0, Xd._h, Y._h))
        if tmp:
            Xd.free()
            y = Y.numpy()
            Y.free()
            if np.ndim(X) == 1:
                y = y[:, 0]
            return y
        return Y

    def __matmul__(self, X):
        return self.apply(X, trans=False)

    def __rmatmul__(self, Bt):
        # `B' * A = (A' * B)'`  (src/lowrank.jl:131-133; RandMatFact.jl:85)
        Bt = np.asarray(Bt, dtype=np.float64)
        return self.apply(np.ascontiguousarray(Bt.T), trans=True).T

    __array_ufunc__ = None

    def free(self):
        if getattr(self, "_h", None) and self._h:
            self._lib.gsi_op_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class _TransposedView:
    __array_ufunc__ = None

    def __init__(self, op):
        self.op = op

    @property
    def shape(self):
        return self.op.shape[::-1]

    @property
    def T(self):
        return self.op

    def __matmul__(self, X):
        return self.op.apply(X, trans=True)


class DenseMatrix(_Operator):
    """A dense `A::Matrix{Float64}` held on the device (column-major, read by TMA).
    On a multi-rank context pass this rank's row block and (row0, m_global)."""

    def __init__(self, A, ctx=None, row0=0, m_global=None):
        super().__init__(ctx or default_context())
        A = _f64_colmajor(A)
        self._buf = DeviceMatrix.from_host(self.ctx, A, LAYOUT_COLMAJOR)
        self.row0, self.mloc = int(row0), A.shape[0]
        m_global = A.shape[0] if m_global is None else int(m_global)
        check(self._lib.gsi_op_dense(self.ctx._h, self._buf._h, self.row0, m_global, C.byref(self._h)))


class LowRankCovMatrix(_Operator):
    """`LowRankCovMatrix(samples)` (reference src/lowrank.jl:14-30): S S'/(N-1) of the
    mean-removed fields; products run as two tensor-core GEMMs."""
    symmetric = True

    def __init__(self, samples, ctx=None, remove_mean=True, row0=0, n_global=None):
        """samples: list of fields or n x N matrix.  Multi-rank context: pass this rank's rows
        samples[row0 : row0 + mloc] and the global field length n_global."""
        super().__init__(ctx or default_context())
        if isinstance(samples, (list, tuple)):
            S = np.stack([np.asarray(s, dtype=np.float64) for s in samples], axis=1)
        else:
            S = np.asarray(samples, dtype=np.float64)
        S = _f64_colmajor(S)
        self.nsamples = S.shape[1]
        self._buf = DeviceMatrix.from_host(self.ctx, S, LAYOUT_COLMAJOR)
        self.row0, self.mloc = int(row0), S.shape[0]
        n_global = S.shape[0] if n_global is None else int(n_global)
        if self.row0 == 0 and n_global == S.shape[0]:
            check(self._lib.gsi_op_lowrankcov(self.ctx._h, self._buf._h, 1 if remove_mean else 0, C.byref(self._h)))
        else:
            check(self._lib.gsi_op_lowrankcov_sharded(self.ctx._h, self._buf._h, 1 if remove_mean else 0, self.row0,
                                                      n_global, C.byref(self._h)))

    @classmethod
    def from_device(cls, samples, remove_mean=True):
        """Wrap an n x N COLMAJOR DeviceMatrix of sample fields that is already on the device (e.g. from
        FFTRF.sample_fields_device); the operator takes the buffer over (its mean is removed in place)."""
        if samples.layout != LAYOUT_COLMAJOR:
            raise ValueError("LowRankCovMatrix.from_device needs a COLMAJOR DeviceMatrix (n x N)")
        self = cls.__new__(cls)
        _Operator.__init__(self, samples.ctx)
        self.nsamples = samples.shape[1]
        self._buf = samples
        self.row0, self.mloc = 0, samples.shape[0]
        check(self._lib.gsi_op_lowrankcov(self.ctx._h, samples._h, 1 if remove_mean else 0, C.byref(self._h)))
        return self


class KernelCovMatrix(_Operator):
    """Matrix-free covariance operator C[i,j] = sigma2*k(|(x_i-x_j)./ell|) + nugget*(i==j)
    (NEW operator type with LowRankCovMatrix's method set; SURVEY.md F4).
    kind: "exponential", "gaussian", "powerlaw", "matern32", "matern52" or "spherical" (or its
    KERNEL_* code; formulas in include/gsi_b200.h).
    coords: d x n (point j = coords[:, j]).  On a multi-rank context this rank applies
    rows [row0, row0+mloc)."""
    symmetric = True

    def __init__(self, kind, coords, ell, sigma2=1.0, nugget=0.0, beta=1.0, ctx=None, row0=0, mloc=None):
        super().__init__(ctx or default_context())
        coords = _f64_colmajor(coords)
        d, n = coords.shape
        ell = np.ascontiguousarray(np.broadcast_to(np.asarray(ell, dtype=np.float64), (d,)))
        self.row0 = int(row0)
        self.mloc = int(n - row0 if mloc is None else mloc)
        self.kind = _KINDS[kind]
        check(self._lib.gsi_op_kernelcov(self.ctx._h, self.kind, d, n, _pd(coords), _pd(ell), float(sigma2),
                                         float(nugget), float(beta), self.row0, self.mloc, C.byref(self._h)))


class GridKernelCovMatrix(_Operator):
    """KernelCovMatrix for points on a structured grid (shape[0] fastest = Julia linear index of
    an array of size `shape`; coordinates idx .* spacing).  A stationary kernel on a lattice has
    only prod(shape) distinct values, which are tabulated once; the product kernel looks them up
    by lattice offset instead of evaluating exp/sqrt on the FP64 pipe it shares with the tensor
    MMAs.  Identical products to KernelCovMatrix(kind, grid_coords(shape) * spacing, ell)."""
    symmetric = True

    def __init__(self, kind, shape, ell, spacing=None, sigma2=1.0, nugget=0.0, beta=1.0, ctx=None, row0=0, mloc=None):
        super().__init__(ctx or default_context())
        shape = [int(s) for s in shape]
        d = len(shape)
        n = int(np.prod(shape))
        dims = (C.c_int64 * d)(*shape)
        spacing = np.ascontiguousarray(np.broadcast_to(np.asarray(1.0 if spacing is None else spacing, dtype=np.float64), (d,)))
        ell = np.ascontiguousarray(np.broadcast_to(np.asarray(ell, dtype=np.float64), (d,)))
        self.row0 = int(row0)
        self.mloc = int(n - row0 if mloc is None else mloc)
        self.kind = _KINDS[kind]
        check(self._lib.gsi_op_kernelcov_grid(self.ctx._h, self.kind, d, dims, _pd(spacing), _pd(ell), float(sigma2),
                                              float(nugget), float(beta), self.row0, self.mloc, C.byref(self._h)))


def rotation_matrix(angles):
    """Rotation R (u = R x) onto the principal axes of an anisotropic structure.  2-D: one angle in radians,
    counter-clockwise from the x axis to the first principal axis.  3-D: three intrinsic z-y-x angles (the first
    about z, the second about the new y, the third about the newest x).  The rows of R are the principal axes."""
    a = np.atleast_1d(np.asarray(angles, dtype=np.float64))
    if a.size == 1:
        c, s = np.cos(a[0]), np.sin(a[0])
        return np.array([[c, s], [-s, c]])
    if a.size != 3:
        raise ValueError("rotation_matrix: one angle (2-D) or three z-y-x angles (3-D)")
    cz, sz = np.cos(a[0]), np.sin(a[0])
    cy, sy = np.cos(a[1]), np.sin(a[1])
    cx, sx = np.cos(a[2]), np.sin(a[2])
    rz = np.array([[cz, -sz, 0.0], [sz, cz, 0.0], [0.0, 0.0, 1.0]])
    ry = np.array([[cy, 0.0, sy], [0.0, 1.0, 0.0], [-sy, 0.0, cy]])
    rx = np.array([[1.0, 0.0, 0.0], [0.0, cx, -sx], [0.0, sx, cx]])
    return (rz @ ry @ rx).T                # columns of rz ry rx: the principal axes in world coordinates


class CovStructure:
    """One structure of a nested covariance model: sill * k_kind(r2), r2 = |(R x_i - R x_j) ./ ranges|^2 (with the
    kind's scaling, include/gsi_b200.h).  rotation: d x d orthonormal R (u = R x, see rotation_matrix) or None."""

    def __init__(self, kind, sill, ranges, rotation=None, beta=1.0):
        self.kind = _KINDS[kind]
        self.sill = float(sill)
        self.ranges = np.atleast_1d(np.asarray(ranges, dtype=np.float64))
        self.rotation = None if rotation is None else np.asarray(rotation, dtype=np.float64)
        self.beta = float(beta)


def _model_args(structures, d):
    """ctypes arguments (nstruct, kinds, sills, ranges, rotations or None, betas) of the gsi_op_kernelcov_model* calls;
    the arrays are returned too, to keep them alive through the call."""
    structures = list(structures)
    ns = len(structures)
    kinds = (C.c_int32 * max(ns, 1))(*[s.kind for s in structures])
    sills = np.array([s.sill for s in structures], dtype=np.float64)
    ranges = np.concatenate([np.broadcast_to(s.ranges, (d,)) for s in structures]) if ns else np.zeros(1)
    ranges = np.ascontiguousarray(ranges, dtype=np.float64)
    betas = np.array([s.beta for s in structures], dtype=np.float64)
    rot = None
    if any(s.rotation is not None for s in structures):
        rot = np.concatenate([(np.eye(d) if s.rotation is None else s.rotation.reshape(d, d)).ravel(order="F")
                              for s in structures])
        rot = np.ascontiguousarray(rot, dtype=np.float64)
    keep = (kinds, sills, ranges, betas, rot)
    args = [ns, kinds, _pd(sills) if ns else None, _pd(ranges), None if rot is None else _pd(rot),
            _pd(betas) if ns else None]
    return args, keep


class KernelCovModelMatrix(_Operator):
    """Matrix-free covariance operator of a nested model (gsi_op_kernelcov_model):
    C[i,j] = sum_s sill_s k_s(x_i, x_j) + nugget (i == j), 1 to MODEL_MAX_STRUCTURES CovStructure terms, each with its
    own kind, ranges and rotation.  coords: d x n.  Several structures are summed inside the product kernel, so the
    model costs one operator application."""
    symmetric = True

    def __init__(self, structures, coords, nugget=0.0, ctx=None, row0=0, mloc=None):
        super().__init__(ctx or default_context())
        coords = _f64_colmajor(coords)
        d, n = coords.shape
        self.row0 = int(row0)
        self.mloc = int(n - row0 if mloc is None else mloc)
        args, self._keep = _model_args(structures, d)
        check(self._lib.gsi_op_kernelcov_model(self.ctx._h, d, n, _pd(coords), *args, float(nugget), self.row0,
                                               self.mloc, C.byref(self._h)))


class GridKernelCovModelMatrix(_Operator):
    """KernelCovModelMatrix for points on a structured grid (as GridKernelCovMatrix): the whole model is tabulated once
    per lattice offset (signed offsets when a structure is rotated)."""
    symmetric = True

    def __init__(self, structures, shape, spacing=None, nugget=0.0, ctx=None, row0=0, mloc=None):
        super().__init__(ctx or default_context())
        shape = [int(s) for s in shape]
        d = len(shape)
        n = int(np.prod(shape))
        dims = (C.c_int64 * d)(*shape)
        spacing = np.ascontiguousarray(np.broadcast_to(np.asarray(1.0 if spacing is None else spacing, dtype=np.float64), (d,)))
        self.row0 = int(row0)
        self.mloc = int(n - row0 if mloc is None else mloc)
        args, self._keep = _model_args(structures, d)
        check(self._lib.gsi_op_kernelcov_model_grid(self.ctx._h, d, dims, _pd(spacing), *args, float(nugget), self.row0,
                                                    self.mloc, C.byref(self._h)))


class KernelCrossCovMatrix(_Operator):
    """Matrix-free cross-covariance C(T, S) of a nested model between targets T (d x m) and sources S (d x n)
    (gsi_op_kernelcov_cross): C[i,j] = sum_s sill_s k_s(t_i, s_j), no nugget.  Kriging / conditioning is C(T, S) w;
    with point observations H, Q H' = C(grid, obs).  Not symmetric: A.T @ X (or X' @ A) is C(S, T) X, on a multi-rank
    context summed over the ranks, each of which owns the target rows [row0, row0 + mloc)."""
    symmetric = False

    def __init__(self, structures, targets, sources, ctx=None, row0=0, mloc=None):
        super().__init__(ctx or default_context())
        targets, sources = _f64_colmajor(targets), _f64_colmajor(sources)
        d, m = targets.shape
        if sources.shape[0] != d:
            raise ValueError(f"KernelCrossCovMatrix: targets are {d}-D, sources {sources.shape[0]}-D")
        n = sources.shape[1]
        self.row0 = int(row0)
        self.mloc = int(m - row0 if mloc is None else mloc)
        args, self._keep = _model_args(structures, d)
        check(self._lib.gsi_op_kernelcov_cross(self.ctx._h, d, m, _pd(targets), n, _pd(sources), *args, self.row0,
                                               self.mloc, C.byref(self._h)))


def _index_array(idx):
    """(count, ctypes int64 array or None) of a list of 0-based linear grid indices (None: every node in order)."""
    if idx is None:
        return None, None
    a = np.ascontiguousarray(np.asarray(idx, dtype=np.int64).ravel())
    return a.size, a


class GridKernelCrossCovMatrix(_Operator):
    """KernelCrossCovMatrix for points that are nodes of one structured grid (as GridKernelCovModelMatrix), given by
    0-based linear indices (shape[0] fastest); targets / sources None: every node in order.  The model is tabulated
    once per lattice offset."""
    symmetric = False

    def __init__(self, structures, shape, targets=None, sources=None, spacing=None, ctx=None, row0=0, mloc=None):
        super().__init__(ctx or default_context())
        shape = [int(s) for s in shape]
        d = len(shape)
        nodes = int(np.prod(shape))
        dims = (C.c_int64 * d)(*shape)
        spacing = np.ascontiguousarray(np.broadcast_to(np.asarray(1.0 if spacing is None else spacing, dtype=np.float64), (d,)))
        m, ti = _index_array(targets)
        n, si = _index_array(sources)
        m = nodes if m is None else m
        n = nodes if n is None else n
        pi64 = C.POINTER(C.c_int64)
        self.row0 = int(row0)
        self.mloc = int(m - row0 if mloc is None else mloc)
        args, keep = _model_args(structures, d)
        self._keep = (keep, ti, si)
        check(self._lib.gsi_op_kernelcov_cross_grid(
            self.ctx._h, d, dims, _pd(spacing), m, None if ti is None else ti.ctypes.data_as(pi64), n,
            None if si is None else si.ctypes.data_as(pi64), *args, self.row0, self.mloc, C.byref(self._h)))


def as_operator(A, ctx=None):
    if isinstance(A, _Operator):
        return A
    if isinstance(A, np.ndarray):
        return DenseMatrix(A, ctx)
    raise TypeError(f"cannot use {type(A).__name__} as an operator: pass an ndarray or a gsi_b200 operator")


def partition_rows(n, world, rank, align=64):
    """Contiguous row block of rank `rank` (blocks are multiples of `align` rows)."""
    per = -(-n // world)
    per = -(-per // align) * align
    r0 = min(n, rank * per)
    r1 = min(n, r0 + per)
    return r0, r1 - r0
