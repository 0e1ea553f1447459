"""grates_b200 -- B200 (sm_100a) implementation of the spherical-harmonic hot path of
akvas/grates: synthesis (``PotentialCoefficients.to_grid``), grid-to-coefficient analysis,
covariance propagation and order-wise filtering, single sets and epoch batches.

Host code is Python (numpy for small tables, torch for device memory / streams /
torch.distributed); all arithmetic on the path runs in hand-written CUDA kernels behind the
C ABI of ``include/grates_b200.h``.  There is no CPU fallback.
"""
from . import _lib, utilities, kernel, plan, grid, gravityfield, filter, distributed, lstsq, io  # noqa: F401
from .gravityfield import PotentialCoefficients, SurfaceMasCons, RadialBasisFunctions, AnisotropicBasisFunctions, TimeSeries, to_grid_batch, gridded_rms, grid_statistics, ravel_batch, gradient_batch, gradient_at_positions  # noqa: F401
from .grid import (RegularGrid, IrregularGrid, GeographicGrid, GaussGrid, analysis_batch, basin_variances,  # noqa: F401
                   covariance_from_normals)
from .filter import OrderWiseFilter, Gaussian, Butterworth, GeneralMatrix, VDK, SpatialFilter  # noqa: F401
from .kernel import get_kernel  # noqa: F401
from .lstsq import BlockMatrix, NormalEquations  # noqa: F401
from .install import install, uninstall, installed  # noqa: F401
from .plan import (SHPlan, PointsPlan, get_plan, get_points_plan, get_gradient_plan, get_gradient_points_plan,  # noqa: F401
                   clear_plan_cache, PinnedArray)

__version__ = "0.1.0"
