"""gsi_b200 -- B200-native randomized low-rank factorization path of
GeostatInversion.jl (RandMatFact.rangefinder / randsvd + covariance products for
pcgalsqr / rga), behind the reference's own function names.

All compute goes through lib/libgsi_b200.so (hand-written sm_100a CUDA).  There is no
CPU fallback: importing works anywhere, creating a Context needs a B200.
"""
from . import _lib
from ._lib import (GsiError, SingularException, PosDefException, DimensionMismatch, NoDeviceError,
                   LAYOUT_TALL, LAYOUT_COLMAJOR, KERNEL_EXPONENTIAL, KERNEL_GAUSSIAN, KERNEL_POWERLAW,
                   KERNEL_MATERN32, KERNEL_MATERN52, KERNEL_SPHERICAL, MODEL_MAX_STRUCTURES, NORMALISER_LU_REF,
                   NORMALISER_QR)
from .core import (Context, DeviceMatrix, DenseMatrix, LowRankCovMatrix, KernelCovMatrix, GridKernelCovMatrix, default_context,
                   set_default_context, as_operator, partition_rows, CovStructure, rotation_matrix, KernelCovModelMatrix,
                   GridKernelCovModelMatrix, KernelCrossCovMatrix, GridKernelCrossCovMatrix)
from . import randmatfact as RandMatFact
from .randmatfact import randsvd, rangefinder, eig_nystrom
from . import dist
from . import fftrf as FFTRF
from .fftrf import PowerLawFieldSampler
from .pcga import (getxis, pcgalsqr, pcgadirect, pcga, rga, PCGALowRankMatrix, lu_L, qr_thinQ, svd_small)
