"""Potential-coefficient containers with GPU synthesis.  Mirrors PotentialCoefficients and
TimeSeries of grates.gravityfield (reference gravityfield.py:76-421, :815-1052) for the hot
path: same packed ``anm`` layout, same ``to_grid(grid, kernel)`` signature and return type;
plus the batched entry points the reference lacks (its users loop over epochs,
gravityfield.py:1143-1172).
"""
import ctypes

import numpy as np
import torch

from . import _lib, plan as _plan, utilities
from .grid import GeographicGrid

GM_DEFAULT = 3.9860044150e+14
R_DEFAULT = 6.3781363000e+06


def degree_indices(n, max_order=None):
    """Packed-array indices of all coefficients of degree n: cosines by increasing order, then
    sines (reference gravityfield.py:15-40)."""
    count = n if max_order is None else min(n, max_order)
    rows = np.concatenate((np.full(count + 1, n, dtype=int), np.arange(count, dtype=int)))
    cols = np.concatenate((np.arange(count + 1, dtype=int), np.full(count, n, dtype=int)))
    return rows, cols


def order_indices(max_degree, m):
    """Packed-array indices of all coefficients of order m (reference gravityfield.py:43-73)."""
    rows = np.arange(m, max_degree + 1, dtype=int)
    cols = np.full(rows.size, m)
    if m > 0:
        rows = np.concatenate((rows, np.full(max_degree + 1 - m, m - 1)))
        cols = np.concatenate((cols, np.arange(m, max_degree + 1, dtype=int)))
    return rows, cols


class PotentialCoefficients:
    """A set of potential coefficients: C_nm = anm[n, m], S_nm = anm[m-1, n]."""

    def __init__(self, GM=GM_DEFAULT, R=R_DEFAULT, max_degree=None):
        self.GM = GM
        self.R = R
        count = 0 if max_degree is None else max_degree + 1
        self.anm = np.zeros((count, count))
        self.epoch = None

    def copy(self):
        gf = PotentialCoefficients(self.GM, self.R)
        gf.anm = self.anm.copy()
        gf.epoch = self.epoch
        return gf

    @property
    def max_degree(self):
        return self.anm.shape[0] - 1

    def truncate(self, max_degree):
        if max_degree < self.max_degree:
            self.anm = self.anm[0:max_degree + 1, 0:max_degree + 1]

    def _degree_array(self):
        idx = np.arange(self.max_degree + 1)
        return np.maximum(idx[:, None], idx[None, :]) * (idx[None, :] > idx[:, None]) + \
            idx[:, None] * (idx[None, :] <= idx[:, None])

    def __add__(self, other):
        if not isinstance(other, PotentialCoefficients):
            raise TypeError("unsupported operand type(s) for +: '" + str(type(self)) + "' and '" + str(type(other)) + "'")
        factor = (other.R / self.R) ** other._degree_array() * (other.GM / self.GM)
        if self.max_degree >= other.max_degree:
            result = self.copy()
            result.anm[0:other.anm.shape[0], 0:other.anm.shape[1]] += other.anm * factor
        else:
            result = PotentialCoefficients(self.GM, self.R)
            result.anm = other.anm * factor
            result.anm[0:self.anm.shape[0], 0:self.anm.shape[1]] += self.anm
            result.epoch = self.epoch
        return result

    def __mul__(self, other):
        if not isinstance(other, (int, float)):
            raise TypeError("unsupported operand type(s) for *: '" + str(type(self)) + "' and '" + str(type(other)) + "'")
        result = self.copy()
        result.anm *= other
        return result

    def __sub__(self, other):
        if not isinstance(other, PotentialCoefficients):
            raise TypeError("unsupported operand type(s) for -: '" + str(type(self)) + "' and '" + str(type(other)) + "'")
        return self + (other * -1)

    def __truediv__(self, other):
        if not isinstance(other, (int, float)):
            raise TypeError("unsupported operand type(s) for /: '" + str(type(self)) + "' and '" + str(type(other)) + "'")
        return self * (1.0 / other)

    @property
    def values(self):
        """Degree-wise ravelled coefficient vector (reference gravityfield.py:392-402)."""
        return utilities.ravel_coefficients(self.anm)

    @values.setter
    def values(self, val):
        if isinstance(val, np.ndarray):
            if val.ndim > 1:
                raise ValueError("unable to assign values of dimension {0:d} to gravity field".format(val.ndim))
            self.anm = utilities.unravel_coefficients(val)
        else:
            raise ValueError("grid values must be either None or " + str(np.ndarray))

    def to_grid(self, grid=None, kernel='ewh'):
        """Gridded values of the coefficient set on a regular grid, computed on the GPU.

        Parameters and return value as reference gravityfield.py:331-390: returns a deep copy
        of ``grid`` (same class) whose values hold the synthesis; the input grid is left
        untouched.  Regular grids (``parallels`` x ``meridians``) take the two-stage tensor-core path,
        any other grid with ``longitude`` / ``latitude`` the point-set kernels (the reference's
        irregular branch, gravityfield.py:370-388).  There is no CPU fallback.
        """
        grid = GeographicGrid() if grid is None else grid
        anm = np.ascontiguousarray(self.anm, dtype=float)[None]
        if not (_plan.is_regular(grid) or (hasattr(grid, "longitude") and hasattr(grid, "latitude"))):
            raise TypeError("grid must expose parallels/meridians or longitude/latitude")
        output_grid = grid.copy()
        if _plan.is_regular(grid):
            p = _plan.get_plan(grid, self.max_degree, kernel, self.GM, self.R)
            output_grid.values = p.synthesis_host(anm).reshape(-1)
        elif hasattr(grid, "longitude") and hasattr(grid, "latitude"):
            p = _plan.get_points_plan(grid, self.max_degree, kernel, self.GM, self.R)
            dev = torch.device("cuda", p.device)
            output_grid.values = p.synthesis(torch.as_tensor(anm).to(dev)).cpu().numpy().reshape(-1)
        else:
            raise TypeError("grid must expose parallels/meridians or longitude/latitude")
        return output_grid


class SurfaceMasCons:
    """Mascon values on a point distribution (reference gravityfield.py:484-570): a container whose analysis runs through
    the point-set kernels (``IrregularGrid.to_potential_coefficients`` -> gb_points_synthesis_matrix) or, for a regular
    grid, the separable analysis kernels."""

    def __init__(self, point_distribution, kernel):
        self.point_distribution = point_distribution
        if self.point_distribution.values is None:
            self.point_distribution.values = np.zeros(self.point_distribution.point_count)
        self.kernel = kernel
        self.epoch = None

    def copy(self):
        other = SurfaceMasCons(self.point_distribution.copy(), self.kernel)
        other.epoch = self.epoch
        return other

    def is_compatible(self, other):
        return self.point_distribution.is_compatible(other.point_distribution)

    @property
    def values(self):
        return self.point_distribution.values

    @values.setter
    def values(self, val):
        self.point_distribution.values = val

    def _checked(self, other, symbol):
        if not isinstance(other, SurfaceMasCons):
            raise TypeError("unsupported operand type(s) for " + symbol + ": '" + str(type(self)) + "' and '" + str(type(other)) + "'")
        if not self.is_compatible(other):
            raise ValueError("point distributions of '" + str(type(self)) + "' instances are not compatible")

    def __add__(self, other):
        self._checked(other, '+')
        result = self.copy()
        result.values = result.values + other.values
        return result

    def __sub__(self, other):
        self._checked(other, '-')
        result = self.copy()
        result.values = result.values - other.values
        return result

    def __mul__(self, other):
        if not isinstance(other, (int, float)):
            raise TypeError("unsupported operand type(s) for *: '" + str(type(self)) + "' and '" + str(type(other)) + "'")
        result = self.copy()
        result.values = result.values * other
        return result

    def __truediv__(self, other):
        if not isinstance(other, (int, float)):
            raise TypeError("unsupported operand type(s) for /: '" + str(type(self)) + "' and '" + str(type(other)) + "'")
        return self * (1.0 / other)

    def to_potential_coefficients(self, min_degree, max_degree, GM=GM_DEFAULT, R=R_DEFAULT):
        """Spherical-harmonic analysis of the mascon values with the instance's kernel.  (The reference passes the builtin
        ``round`` where R belongs, gravityfield.py:570, and fails; R is passed here.)"""
        out = self.point_distribution.to_potential_coefficients(min_degree, max_degree, self.kernel, GM, R)
        out.epoch = self.epoch
        return out


class AnisotropicBasisFunctions:
    """Gravity field represented by anisotropic kernel basis functions (reference gravityfield.py:573-642).

    ``to_grid`` in the reference is ``K @ (Y' v)`` accumulated over 512-point blocks, followed by a synthesis that loops
    over the meridians.  Here: the point-set adjoint (``gb_points_adjoint``, unit degree factors), the dense matrix on the
    filter GEMM (``gb_dense_filter``), and the regular-grid synthesis -- three device calls, no table ever on the host.
    """

    def __init__(self, point_distribution, K, min_degree, max_degree, GM=GM_DEFAULT, R=R_DEFAULT):
        self._K = np.array(K, dtype=float, copy=True)
        self.point_distribution = point_distribution
        self._min_degree = min_degree
        self._max_degree = max_degree
        self.GM = GM
        self.R = R
        self.epoch = None
        self.values = np.zeros((self.point_distribution.size))
        self._operator = None
        self._plan_cache = None

    @property
    def values(self):
        return self.point_distribution.values

    @values.setter
    def values(self, val):
        self.point_distribution.values = val

    def is_compatible(self, other):
        return self.point_distribution.is_compatible(other.point_distribution)

    def to_potential_coefficients_batch(self, values):
        """values [E, points] (numpy or CUDA tensor) -> CUDA tensor [E, L, L]: unravel(K @ ravel(Y' v)), degrees below
        the minimum degree zero."""
        from .filter import GeneralMatrix
        grid = self.point_distribution
        lon = np.asarray(grid.longitude, dtype=float)
        lat = np.asarray(grid.latitude, dtype=float)
        key = (lon.tobytes(), lat.tobytes(), float(grid.semimajor_axis), float(grid.flattening))
        if self._plan_cache is None or self._plan_cache[0] != key:
            ones = np.ones((lon.size, self._max_degree + 1))
            self._plan_cache = (key, _plan.PointsPlan(lon, lat, grid.semimajor_axis, grid.flattening, self._max_degree,
                                                      degree_factors=ones))
        p = self._plan_cache[1]
        if self._operator is None:
            self._operator = GeneralMatrix(self._K, self._min_degree, self._max_degree)
        dev = torch.device("cuda", p.device)
        v = values if isinstance(values, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(values, dtype=float))
        anm = self._operator.filter_batch(p.adjoint(v.to(dev)))
        anm[:, 0:self._min_degree, 0:self._min_degree] = 0.0        # the dense operator passes lower degrees through
        return anm

    def to_grid(self, grid=None, kernel='ewh'):
        grid = GeographicGrid() if grid is None else grid
        anm = self.to_potential_coefficients_batch(np.asarray(self.values, dtype=float)[None])
        output_grid = grid.copy()
        output_grid.values = to_grid_batch(anm, grid, kernel, self.GM, self.R)[0].cpu().numpy().reshape(-1)
        return output_grid


class RadialBasisFunctions:
    """Gravity field represented by radial basis functions at nodal points (reference gravityfield.py:645-781).

    Constructor, ``values``, ``copy`` and ``to_grid`` as in the reference.  ``to_potential_coefficients`` runs the sum
    over the nodal points as one GEMM against the on-the-fly design matrix (``gb_points_adjoint``); ``blocking_factor``
    is accepted for signature compatibility and ignored (the device code blocks by itself).
    """

    def __init__(self, point_distribution, K, min_degree, max_degree, GM=GM_DEFAULT, R=R_DEFAULT):
        self._K = np.array(K, dtype=float, copy=True)
        self.point_distribution = point_distribution.copy()
        self._min_degree = min_degree
        self._max_degree = max_degree
        self.GM = GM
        self.R = R
        self.epoch = None
        self.values = np.zeros((self.point_distribution.size))

    def copy(self):
        rbf = RadialBasisFunctions(self.point_distribution.copy(), self._K, self._min_degree, self._max_degree, self.GM, self.R)
        rbf.epoch = self.epoch
        rbf.values = self.values.copy()
        return rbf

    @property
    def values(self):
        return self.point_distribution.values

    @values.setter
    def values(self, val):
        self.point_distribution.values = val

    def is_compatible(self, other):
        return self.point_distribution.is_compatible(other.point_distribution)

    def _points_plan(self):
        """Point-set plan whose degree factors are the upward continuation (R / r_p)^(n + 1), gravityfield.py:713."""
        grid = self.point_distribution
        lon = np.asarray(grid.longitude, dtype=float)
        lat = np.asarray(grid.latitude, dtype=float)
        key = (lon.tobytes(), lat.tobytes(), float(grid.semimajor_axis), float(grid.flattening), self._max_degree, float(self.R))
        cached = getattr(self, "_plan_cache", None)
        if cached is None or cached[0] != key:
            radius = utilities.geocentric_radius(lat, grid.semimajor_axis, grid.flattening)
            kn = np.power((self.R / radius)[:, np.newaxis], np.arange(self._max_degree + 1, dtype=int) + 1)
            cached = (key, _plan.PointsPlan(lon, lat, grid.semimajor_axis, grid.flattening, self._max_degree,
                                            degree_factors=kn))
            self._plan_cache = cached
        return cached[1]

    def to_potential_coefficients_batch(self, values):
        """values [E, points] (numpy or CUDA tensor) -> CUDA tensor [E, L, L] of packed coefficients."""
        p = self._points_plan()
        dev = torch.device("cuda", p.device)
        v = values if isinstance(values, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(values, dtype=float))
        anm = p.adjoint(v.to(dev))
        return anm.mul_(torch.as_tensor(self._K).to(dev))

    def to_potential_coefficients(self, blocking_factor=256):
        coefficients = PotentialCoefficients(self.GM, self.R)
        coefficients.anm = self.to_potential_coefficients_batch(np.asarray(self.values, dtype=float)[None])[0].cpu().numpy()
        coefficients.epoch = self.epoch
        return coefficients

    def to_potential_coefficients_matrix(self, blocking_factor=256):
        """Matrix [K', points] from the radial basis function coefficients to degree-wise ordered spherical harmonics
        (reference gravityfield.py:729-763): the transposed point-set design matrix scaled by the shape factors."""
        A = self._points_plan().synthesis_matrix(self._min_degree)
        k = torch.as_tensor(utilities.ravel_coefficients(self._K, self._min_degree, self._max_degree)).to(A.device)
        return (A * k[None, :]).T.contiguous().cpu().numpy()

    def to_grid(self, grid=None, kernel='ewh'):
        return self.to_potential_coefficients().to_grid(GeographicGrid() if grid is None else grid, kernel)


class TimeSeries:
    """Epoch-sorted list of gravity fields (reference gravityfield.py:815-1052)."""

    def __init__(self, data):
        self._data = list(data)
        self._dtype = type(self._data[0])
        for d in self._data:
            if not isinstance(d, self._dtype):
                raise ValueError("Found inconsistent data types (" + str(self._dtype) + " and " + str(type(d)) + ")")
            if d.epoch is None:
                raise ValueError("At least one data point has no valid time stamp")
        self.sort()

    def __len__(self):
        return len(self._data)

    def __getitem__(self, index):
        return self._data[index]

    def sort(self):
        self._data.sort(key=lambda d: d.epoch)

    def items(self):
        for d in self._data:
            yield d.epoch, d

    def epochs(self):
        return [d.epoch for d in self._data]

    def copy(self):
        return TimeSeries([d.copy() for d in self._data])

    def interpolate_to(self, epoch):
        """Piecewise linear interpolation to an epoch inside the series (reference
        gravityfield.py:915-946); extrapolation raises ValueError."""
        t = np.array([d.epoch for d in self._data])
        if t.size < 2:
            raise ValueError("at least two data points are required for interpolation")
        if epoch < t[0] or epoch > t[-1]:
            raise ValueError("extrapolation is not supported (trying to extrapolate to " + str(epoch) +
                             " from the interval " + str(t[0]) + ", " + str(t[-1]) + ")")
        idx = max(int(np.searchsorted(t, epoch)), 1)
        weight = (epoch - t[idx - 1]).total_seconds() / (t[idx] - t[idx - 1]).total_seconds()
        output = self._data[idx - 1] * (1 - weight) + self._data[idx] * weight
        output.epoch = epoch
        return output

    def evaluate_at(self, epoch):
        return self.interpolate_to(epoch)

    def to_array(self):
        """[epochs, (N+1)^2] matrix in degree-wise order (reference gravityfield.py:964-980)."""
        width = self._data[0].values.size
        return np.stack([d.values[0:width] for d in self._data])

    def to_array_device(self, min_degree=0):
        """Same matrix as ``to_array`` (from ``min_degree`` on) as a CUDA tensor [epochs, K']: the packed batch is
        uploaded once and ravelled on the GPU (gb_ravel_coefficients), the form the covariance / filter-matrix
        entry points consume."""
        return ravel_batch(self.to_packed(), min_degree)

    def to_packed(self):
        """[epochs, L, L] packed coefficient array (zero-padded to the largest degree)."""
        L = max(d.anm.shape[0] for d in self._data)
        out = np.zeros((len(self._data), L, L))
        for k, d in enumerate(self._data):
            out[k, :d.anm.shape[0], :d.anm.shape[1]] = d.anm
        return out

    def to_grid(self, grid=None, kernel='ewh', device_output=False, out=None):
        """Synthesis of the whole series in one batched GPU call -> [epochs, nlat, nlon]
        (numpy, or a CUDA tensor with ``device_output=True``)."""
        first = self._data[0]
        for d in self._data:
            if d.GM != first.GM or d.R != first.R:
                raise ValueError("all epochs of a batched synthesis must share GM and R")
        return to_grid_batch(self.to_packed(), grid, kernel, first.GM, first.R, device_output=device_output, out=out)


def ravel_batch(anm, min_degree=0):
    """Packed [E, L, L] coefficients (numpy or CUDA tensor) -> degree-wise vectors [E, (N+1)^2 - min_degree^2] on the
    device (reference utilities.py:310-360 for a whole batch)."""
    on_host = not isinstance(anm, torch.Tensor)
    dev = _plan._current_device(None if on_host else anm.device)
    x = torch.as_tensor(np.ascontiguousarray(anm, dtype=float)).to(torch.device("cuda", dev)) if on_host else anm.contiguous()
    if x.dim() != 3 or x.shape[1] != x.shape[2] or x.dtype != torch.float64:
        raise ValueError("coefficients must be a float64 array of shape [epochs, L, L]")
    nmax = x.shape[-1] - 1
    if not 0 <= min_degree <= nmax:
        raise ValueError("min_degree must lie in [0, {0}]".format(nmax))
    out = torch.empty((x.shape[0], (nmax + 1) ** 2 - min_degree ** 2), dtype=torch.float64, device=x.device)
    _lib.check(_lib.load().gb_ravel_coefficients(ctypes.c_void_p(x.data_ptr()), x.shape[0], nmax, int(min_degree),
                                                 ctypes.c_void_p(out.data_ptr()), dev, _plan._stream_handle(dev)))
    return out


def to_grid_batch(anm, grid=None, kernel='ewh', GM=GM_DEFAULT, R=R_DEFAULT, device_output=False, out=None,
                  degree_weights=None, orderwise_filter=None):
    """Batched synthesis.  anm: [E, L, L] packed coefficients (numpy array or CUDA float64
    tensor).  Returns [E, nlat, nlon]; with a CUDA tensor input (or device_output=True) the
    result stays on the device, otherwise it is copied to the host inside the call.
    degree_weights: weights of an isotropic filter (``Gaussian(r).degree_weights(nmax)``) fused into
    the synthesis on regular grids."""
    grid = GeographicGrid() if grid is None else grid
    L = anm.shape[-1]
    if degree_weights is not None or orderwise_filter is not None:
        # orderwise_filter: an OrderWiseFilter applied first, its result written straight into the synthesis workspace
        if not _plan.is_regular(grid):
            raise ValueError("filters are fused into the regular-grid synthesis only; filter the coefficients first")
        p = _plan.get_plan(grid, L - 1, kernel, GM, R)
        on_device = isinstance(anm, torch.Tensor)
        x = anm if on_device else torch.as_tensor(np.ascontiguousarray(anm, dtype=float)).to(torch.device("cuda", p.device))
        vals = p.synthesis(x, out=out if (on_device or device_output) else None, degree_weights=degree_weights,
                           orderwise_filter=orderwise_filter)
        return vals if (on_device or device_output) else vals.cpu().numpy()
    if not _plan.is_regular(grid):
        p = _plan.get_points_plan(grid, L - 1, kernel, GM, R)      # -> [E, points]
        on_device = isinstance(anm, torch.Tensor)
        x = anm if on_device else torch.as_tensor(np.ascontiguousarray(anm, dtype=float)).to(torch.device("cuda", p.device))
        vals = p.synthesis(x, out=out if on_device or device_output else None)
        return vals if (on_device or device_output) else vals.cpu().numpy()
    p = _plan.get_plan(grid, L - 1, kernel, GM, R)
    if isinstance(anm, torch.Tensor):
        return p.synthesis(anm, out=out)
    if device_output:
        dev = torch.device("cuda", p.device)
        return p.synthesis(torch.as_tensor(np.ascontiguousarray(anm, dtype=float)).to(dev), out=out)
    return p.synthesis_host(anm, out=out)


_FRAMES = ('cartesian', 'local')


def _gradient_input(anm, frame):
    """Checks that need no device: the frame name, the shape [E, L, L] and, for a tensor, float64 on a CUDA device."""
    if frame not in _FRAMES:
        raise ValueError("frame must be 'cartesian' or 'local' (got {0!r})".format(frame))
    x = anm if isinstance(anm, torch.Tensor) else np.ascontiguousarray(anm, dtype=float)
    if x.ndim != 3 or x.shape[1] != x.shape[2]:
        raise ValueError("coefficients must have shape [epochs, L, L] (got {0})".format(tuple(x.shape)))
    if isinstance(x, torch.Tensor) and (x.dtype != torch.float64 or not x.is_cuda):
        raise ValueError("coefficients must be a float64 CUDA tensor")
    return x


# order of the derivative -> (components, coefficient transform, rotation to the local frame)
_DERIVATIVE_CALLS = {1: (3, "gb_gradient_coefficients", "gb_rotate_to_local"),
                     2: (6, "gb_gravity_gradient_coefficients", "gb_rotate_tensor_to_local")}


def _gradient(x, p, frame, shape, device_output, out, order=1):
    """Transform (gb_gradient_coefficients, or gb_gravity_gradient_coefficients for order 2), one synthesis of the C*E
    sets on the plan p of that order, and for frame='local' the rotation (gb_rotate_to_local / gb_rotate_tensor_to_local)
    -> [E, C, *shape] with C = 3 (order 1) or 6 (order 2) components."""
    ncomp, transform, rotation = _DERIVATIVE_CALLS[order]
    on_device = isinstance(x, torch.Tensor)
    dev = torch.device("cuda", p.device)
    if on_device and x.device.index != p.device:
        raise ValueError("coefficients must be a float64 CUDA tensor on device {0}".format(p.device))
    x = x.contiguous() if on_device else torch.as_tensor(x).to(dev)
    E, L = x.shape[0], x.shape[-1]
    full = (E, ncomp) + tuple(shape)
    to_host = not (on_device or device_output)
    if out is not None and to_host:
        _plan._check_out_host(out, full)
    if out is not None and not to_host:
        res = _plan._check_out(out, full, p.device)
    else:
        res = torch.empty(full, dtype=torch.float64, device=dev)
    lib, st = _lib.load(), _plan._stream_handle(p.device)
    Lo = L + order
    g = torch.empty((E, ncomp, Lo, Lo), dtype=torch.float64, device=dev)
    _lib.check(getattr(lib, transform)(ctypes.c_void_p(x.data_ptr()), E, L - 1, ctypes.c_void_p(g.data_ptr()),
                                       p.device, st))
    p.synthesis(g.view(ncomp * E, Lo, Lo), out=res.view((ncomp * E,) + tuple(shape)))
    if frame == 'local':
        _lib.check(getattr(lib, rotation)(ctypes.c_void_p(res.data_ptr()), ctypes.c_void_p(p.frame.data_ptr()), E,
                                          int(np.prod(shape)), p.device, st))
    if not to_host:
        return res
    if out is None:
        return res.cpu().numpy()
    torch.from_numpy(out).copy_(res)
    return out


def gradient_batch(anm, grid=None, GM=GM_DEFAULT, R=R_DEFAULT, frame='cartesian', device_output=False, out=None):
    """Gravitational acceleration grad V of a batch of coefficient sets on a grid, in m/s^2.

    anm: [E, L, L] packed coefficients (numpy array or CUDA float64 tensor).  Returns [E, 3, nlat, nlon] on a regular
    grid, [E, 3, points] on a grid with longitude / latitude (IrregularGrid), at the geocentric radius of the ellipsoid.
    frame='cartesian': components (x, y, z) Earth-fixed; frame='local': (east, north, up) of the GEOCENTRIC SPHERICAL
    frame at each point (up along the geocentric radius, not the ellipsoidal normal).  The gradient of the potential
    only: no kernel and no centrifugal term.  Host / device behaviour as ``to_grid_batch``: with a CUDA tensor input
    (or device_output=True) the result is a CUDA tensor, otherwise a numpy array (``out`` of the matching kind).

    Each component is a scalar synthesis at degree N + 1 of linearly transformed coefficients (Cunningham's relation,
    gb_gradient_coefficients), so the 3E sets run through the same synthesis kernels as ``to_grid_batch``."""
    return _derivative_on_grid(anm, grid, GM, R, frame, device_output, out, 1)


def _derivative_on_grid(anm, grid, GM, R, frame, device_output, out, order):
    x = _gradient_input(anm, frame)
    grid = GeographicGrid() if grid is None else grid
    if _plan.is_regular(grid):
        p = _plan._derivative_plan(grid, x.shape[-1] - 1, order, GM, R, None)
        shape = (p.nlat, p.nlon)
    elif hasattr(grid, "longitude") and hasattr(grid, "latitude"):
        lon = np.asarray(grid.longitude, dtype=float)
        lat = np.asarray(grid.latitude, dtype=float)
        a, f = grid.semimajor_axis, grid.flattening
        p = _plan._derivative_points_plan(utilities.geocentric_radius(lat, a, f), utilities.colatitude(lat, a, f), lon,
                                          x.shape[-1] - 1, order, GM, R, None, True)
        shape = (p.npts,)
    else:
        raise TypeError("grid must expose parallels/meridians or longitude/latitude")
    return _gradient(x, p, frame, shape, device_output, out, order)


def gradient_at_positions(anm, positions, GM=GM_DEFAULT, R=R_DEFAULT, frame='cartesian', device_output=False, out=None):
    """Gravitational acceleration grad V of a batch of coefficient sets at Earth-fixed Cartesian positions [P, 3] in
    metres (any radius, e.g. along an orbit) -> [E, 3, P] in m/s^2.  frame, the result's kind and ``out`` as for
    ``gradient_batch``; the local frame is geocentric spherical at each position (longitude 0 on the polar axis).
    Non-finite positions and the origin raise ValueError."""
    return _derivative_at_positions(anm, positions, GM, R, frame, device_output, out, 1)


def _derivative_at_positions(anm, positions, GM, R, frame, device_output, out, order):
    x = _gradient_input(anm, frame)
    r, colat, lon = utilities.cartesian_to_spherical(positions)
    p = _plan._derivative_points_plan(r, colat, lon, x.shape[-1] - 1, order, GM, R, None, True)
    return _gradient(x, p, frame, (p.npts,), device_output, out, order)


def gravity_gradient_batch(anm, grid=None, GM=GM_DEFAULT, R=R_DEFAULT, frame='cartesian', device_output=False,
                           out=None):
    """Gravity gradient tensor (the second derivatives of the potential) of a batch of coefficient sets on a grid, in
    s^-2 (1 E = 1 Eotvos = 1e-9 s^-2).

    anm: [E, L, L] packed coefficients (numpy array or CUDA float64 tensor).  Returns the upper triangle of the
    symmetric tensor, [E, 6, nlat, nlon] on a regular grid, [E, 6, points] on a grid with longitude / latitude, at the
    geocentric radius of the ellipsoid.  frame='cartesian': (xx, xy, xz, yy, yz, zz) Earth-fixed; frame='local':
    (ee, en, eu, nn, nu, uu) of Q V Q' in (east, north, up) of the geocentric spherical frame, as for ``gradient_batch``.
    The potential only: no kernel and no centrifugal term.  The result's kind and ``out`` as for ``gradient_batch``.

    Component (a, b) is a scalar synthesis at degree N + 2 of the coefficients transformed twice by Cunningham's
    relation (gb_gravity_gradient_coefficients), so the 6E sets run through one synthesis on the same kernels as
    ``to_grid_batch``; no 1 / sin(theta) is involved, so the poles are regular."""
    return _derivative_on_grid(anm, grid, GM, R, frame, device_output, out, 2)


def gravity_gradient_at_positions(anm, positions, GM=GM_DEFAULT, R=R_DEFAULT, frame='cartesian', device_output=False,
                                  out=None):
    """Gravity gradient tensor of a batch of coefficient sets at Earth-fixed Cartesian positions [P, 3] in metres (any
    radius, e.g. along an orbit) -> [E, 6, P] in s^-2 (1 E = 1e-9 s^-2).  Components, frame, the result's kind and
    ``out`` as for ``gravity_gradient_batch``; the local frame as for ``gradient_at_positions``.  Non-finite positions
    and the origin raise ValueError."""
    return _derivative_at_positions(anm, positions, GM, R, frame, device_output, out, 2)


def _gradient_covariance_input(covariance_matrix, min_degree, max_degree, frame, full):
    """Checks that need no device: the frame name, full, the degree range and the shape of Sigma."""
    if frame not in _FRAMES:
        raise ValueError("frame must be 'cartesian' or 'local' (got {0!r})".format(frame))
    if not isinstance(full, (bool, np.bool_)):
        raise ValueError("full must be True or False (got {0!r})".format(full))
    if not 0 <= int(min_degree) <= int(max_degree):
        raise ValueError("degree range [{0}, {1}] is empty or negative".format(min_degree, max_degree))
    kp = (int(max_degree) + 1) ** 2 - int(min_degree) ** 2
    if tuple(np.shape(covariance_matrix)) != (kp, kp):
        raise ValueError("covariance matrix must have shape [{0}, {0}] for degrees {1}..{2} (got {3})".format(
            kp, min_degree, max_degree, tuple(np.shape(covariance_matrix))))


def _gradient_covariance(covariance_matrix, p, min_degree, frame, full, device_output):
    from .grid import _device_matrix
    out = p.gradient_covariance(_device_matrix(covariance_matrix, p.device), int(min_degree), frame, bool(full))
    return out if device_output else out.cpu().numpy()


def gradient_covariance_propagation(covariance_matrix, grid, min_degree, max_degree, GM=GM_DEFAULT, R=R_DEFAULT,
                                    frame='cartesian', full=False, device_output=False):
    """Uncertainty of the gravitational acceleration grad V on a grid, given the covariance matrix Sigma [K', K'] of the
    degree-wise coefficients from min_degree to max_degree (numpy array or CUDA tensor; contracted as its symmetric part
    (Sigma + Sigma') / 2).  Points at the geocentric radius of the ellipsoid, as ``gradient_batch``; frame as there.

    Returns standard deviations in m/s^2, [3, points] on a grid with longitude / latitude and [3, nlat, nlon] on a
    regular grid (its points row by row), or with full=True the 3 x 3 covariances in (m/s^2)^2, [points, 3, 3] or
    [nlat, nlon, 3, 3].  numpy arrays, or CUDA tensors with device_output=True.  Work: 3 P K'^2 flops executed
    (gb_points_gradient_covariance, the lower triangle of the symmetric part)."""
    _gradient_covariance_input(covariance_matrix, min_degree, max_degree, frame, full)
    if _plan.is_regular(grid):
        parallels = np.asarray(grid.parallels, dtype=float)
        meridians = np.asarray(grid.meridians, dtype=float)
        lat, lon = np.repeat(parallels, meridians.size), np.tile(meridians, parallels.size)
        shape = (parallels.size, meridians.size)
    elif hasattr(grid, "longitude") and hasattr(grid, "latitude"):
        lat, lon = np.asarray(grid.latitude, dtype=float), np.asarray(grid.longitude, dtype=float)
        shape = None
    else:
        raise TypeError("grid must expose parallels/meridians or longitude/latitude")
    a, f = grid.semimajor_axis, grid.flattening
    p = _plan.get_gradient_points_plan(utilities.geocentric_radius(lat, a, f), utilities.colatitude(lat, a, f), lon,
                                       int(max_degree), GM, R)
    out = _gradient_covariance(covariance_matrix, p, min_degree, frame, full, device_output)
    if shape is None:
        return out
    return out.reshape(shape + (3, 3)) if full else out.reshape((3,) + shape)


def gradient_covariance_at_positions(covariance_matrix, positions, min_degree, max_degree, GM=GM_DEFAULT, R=R_DEFAULT,
                                     frame='cartesian', full=False, device_output=False):
    """``gradient_covariance_propagation`` at Earth-fixed Cartesian positions [P, 3] in metres (any radius, e.g. along an
    orbit; the local frame as for ``gradient_at_positions``) -> [3, P] standard deviations in m/s^2, or [P, 3, 3]
    covariances in (m/s^2)^2 with full=True.  Non-finite positions and the origin raise ValueError."""
    _gradient_covariance_input(covariance_matrix, min_degree, max_degree, frame, full)
    r, colat, lon = utilities.cartesian_to_spherical(positions)
    p = _plan.get_gradient_points_plan(r, colat, lon, int(max_degree), GM, R)
    return _gradient_covariance(covariance_matrix, p, min_degree, frame, full, device_output)


def _host_or_cuda(x, name):
    """numpy float64 array, or the tensor itself when it is a float64 CUDA tensor."""
    if isinstance(x, torch.Tensor):
        if x.dtype != torch.float64 or not x.is_cuda:
            raise ValueError("{0} must be a float64 CUDA tensor".format(name))
        return x
    return np.asarray(x, dtype=float)


def gradient_adjoint_at_positions(values, positions, max_degree, GM=GM_DEFAULT, R=R_DEFAULT, frame='cartesian',
                                  device_output=False):
    """Transpose of ``gradient_at_positions``: values [E, 3, P] in m/s^2 at Earth-fixed Cartesian positions [P, 3] in
    metres, components in ``frame`` -> packed coefficients [E, L, L], L = max_degree + 1, with
    <gradient_at_positions(X), Y> = <X, gradient_adjoint_at_positions(Y)>: the operator J' of an iterative
    least-squares solver.  With a CUDA tensor input (or device_output=True) the result is a CUDA tensor, otherwise a
    numpy array.  Non-finite positions and the origin raise ValueError."""
    return _derivative_adjoint_at_positions(values, positions, max_degree, GM, R, frame, device_output, 1)


def gravity_gradient_adjoint_at_positions(values, positions, max_degree, GM=GM_DEFAULT, R=R_DEFAULT, frame='cartesian',
                                          device_output=False):
    """Transpose of ``gravity_gradient_at_positions``: values [E, 6, P] in s^-2 at Earth-fixed Cartesian positions [P, 3]
    in metres, the six components (xx, xy, xz, yy, yz, zz) or (ee, en, eu, nn, nu, uu) of ``frame`` -> packed
    coefficients [E, L, L], L = max_degree + 1, with
    <gravity_gradient_at_positions(X), Y> = <X, gravity_gradient_adjoint_at_positions(Y)>.  The result's kind as for
    ``gradient_adjoint_at_positions``.  Non-finite positions and the origin raise ValueError."""
    return _derivative_adjoint_at_positions(values, positions, max_degree, GM, R, frame, device_output, 2)


def _derivative_adjoint_at_positions(values, positions, max_degree, GM, R, frame, device_output, order):
    ncomp = _DERIVATIVE_CALLS[order][0]
    if frame not in _FRAMES:
        raise ValueError("frame must be 'cartesian' or 'local' (got {0!r})".format(frame))
    if int(max_degree) < 0:
        raise ValueError("max_degree must be >= 0 (got {0})".format(max_degree))
    v = _host_or_cuda(values, "values")
    r, colat, lon = utilities.cartesian_to_spherical(positions)
    if v.ndim != 3 or v.shape[1] != ncomp or v.shape[2] != r.size:
        raise ValueError("values must have shape [sets, {0}, {1}] (got {2})".format(ncomp, r.size, tuple(v.shape)))
    p = _plan._derivative_points_plan(r, colat, lon, int(max_degree), order, GM, R, None, True)
    on_device = isinstance(v, torch.Tensor)
    if on_device and v.device.index != p.device:
        raise ValueError("values must be a float64 CUDA tensor on device {0}".format(p.device))
    x = v if on_device else torch.as_tensor(np.ascontiguousarray(v)).to(torch.device("cuda", p.device))
    out = p._derivative_adjoint(x, frame, order)
    return out if (on_device or device_output) else out.cpu().numpy()


def _positions_per_chunk(max_degree, order=1):
    """Positions whose point-plan tables (four [P, N + order + 1] tables) take about 1 GB."""
    return max(1, (1 << 30) // (8 * 4 * (int(max_degree) + order + 1)))


def gradient_normal_equations_at_positions(observations, positions, min_degree, max_degree, GM=GM_DEFAULT, R=R_DEFAULT,
                                           frame='cartesian', weights=None, block_size=2048, positions_per_chunk=None):
    """Least-squares normal equations of gravitational-acceleration observations at Earth-fixed Cartesian positions (the
    acceleration approach of orbit-based gravity recovery), for the degree-wise coefficients from min_degree to
    max_degree, K' = (max_degree + 1)^2 - min_degree^2 unknowns.

    observations: [E, 3, P] or [3, P] in m/s^2 (numpy or CUDA float64), E sets on the same positions sharing one normal
    matrix; components in ``frame`` ('cartesian' (x, y, z), or 'local' (east, north, up) as in ``gradient_at_positions``).
    positions: [P, 3] in metres.  weights: [3, P] positive weights (inverse variances) per observation, or None for 1.
    With J~ the design matrix of grad V (the Jacobian of ``gradient_at_positions`` in ``frame``) and W = diag(weights):

      matrix                  N = J~' W J~ as a device ``lstsq.BlockMatrix`` with blocks of block_size
      right_hand_side         n = J~' W l, CUDA tensor [K', E]
      observation_square_sum  l' W l per set, numpy [E]
      observation_count       3 P

    returned as an ``lstsq.NormalEquations`` (``solve()``, ``compute_covariance()``).  Everything is formed on the device
    (gb_points_gradient_normals, ``gradient_adjoint_at_positions``); long position arrays are cut into chunks of
    positions_per_chunk (None: the positions whose tables take about 1 GB) with point plans of their own, closed after
    use.  Work: about 3 P K'^2 flops on the FP64 tensor cores (the upper triangle of N)."""
    return _normal_equations_at_positions(observations, positions, min_degree, max_degree, GM, R, frame, weights,
                                          block_size, positions_per_chunk, 1)


def gravity_gradient_normal_equations_at_positions(observations, positions, min_degree, max_degree, GM=GM_DEFAULT,
                                                   R=R_DEFAULT, frame='cartesian', weights=None, block_size=2048,
                                                   positions_per_chunk=None):
    """Least-squares normal equations of gravity-gradient observations (a gradiometer) at Earth-fixed Cartesian
    positions, for the degree-wise coefficients from min_degree to max_degree, K' = (max_degree + 1)^2 - min_degree^2
    unknowns.

    observations: [E, 6, P] or [6, P] in s^-2 (numpy or CUDA float64, finite), E sets on the same positions sharing one
    normal matrix; the components (xx, xy, xz, yy, yz, zz) Earth-fixed, or (ee, en, eu, nn, nu, uu) with frame='local',
    as in ``gravity_gradient_at_positions``.  positions: [P, 3] in metres.  weights: [6, P] finite, non-negative weights
    (inverse variances) per observation, or None for 1; a zero weight leaves the observation out (a component the
    instrument measures badly).  With J~ the design matrix of the tensor in ``frame`` and W = diag(weights):

      matrix                  N = J~' W J~ as a device ``lstsq.BlockMatrix`` with blocks of block_size
      right_hand_side         n = J~' W l, CUDA tensor [K', E]
      observation_square_sum  l' W l per set, numpy [E]
      observation_count       the number of positive weights (6 P without weights)

    returned as an ``lstsq.NormalEquations``.  Everything is formed on the device (gb_points_gravity_gradient_normals,
    ``gravity_gradient_adjoint_at_positions``), in chunks of positions as ``gradient_normal_equations_at_positions``.
    Work: about 6 P K'^2 flops on the FP64 tensor cores (the upper triangle of N)."""
    return _normal_equations_at_positions(observations, positions, min_degree, max_degree, GM, R, frame, weights,
                                          block_size, positions_per_chunk, 2)


def _finite(x):
    return bool((torch.isfinite(x) if isinstance(x, torch.Tensor) else np.isfinite(x)).all())


# order of the derivative -> the uncached point plan of the chunks
_CHUNK_PLANS = {1: _plan.gradient_points_plan, 2: _plan.gravity_gradient_points_plan}


def _normal_equations_at_positions(observations, positions, min_degree, max_degree, GM, R, frame, weights, block_size,
                                   positions_per_chunk, order):
    """The normal equations of observations of the derivatives of order 1 (grad V, three components per position, with
    positive weights) or 2 (the gravity gradient tensor, six components, with non-negative weights and finite
    observations): every check before any device work, then the chunks of positions."""
    from .lstsq import BlockMatrix, NormalEquations
    ncomp = _DERIVATIVE_CALLS[order][0]
    if frame not in _FRAMES:
        raise ValueError("frame must be 'cartesian' or 'local' (got {0!r})".format(frame))
    nmin, nmax = int(min_degree), int(max_degree)
    if not 0 <= nmin <= nmax:
        raise ValueError("degree range [{0}, {1}] is empty or negative".format(min_degree, max_degree))
    if int(block_size) < 1:
        raise ValueError("block_size must be positive (got {0})".format(block_size))
    if positions_per_chunk is not None and int(positions_per_chunk) < 1:
        raise ValueError("positions_per_chunk must be positive (got {0})".format(positions_per_chunk))
    obs = _host_or_cuda(observations, "observations")
    w = None if weights is None else _host_or_cuda(weights, "weights")
    r, colat, lon = utilities.cartesian_to_spherical(positions)
    P = r.size
    single = obs.ndim == 2
    if single:
        obs = obs[None]
    if obs.ndim != 3 or obs.shape[1] != ncomp or obs.shape[2] != P or obs.shape[0] < 1:
        raise ValueError("observations must have shape [sets, {0}, {1}] or [{0}, {1}] (got {2})".format(
            ncomp, P, tuple(np.shape(observations))))
    if order == 2 and not _finite(obs):
        raise ValueError("observations must be finite")
    count = ncomp * P
    if w is not None:
        if tuple(w.shape) != (ncomp, P):
            raise ValueError("weights must have shape [{0}, {1}] (got {2})".format(ncomp, P, tuple(w.shape)))
        if order == 1 and not (_finite(w) and bool((w > 0).all())):
            raise ValueError("weights must be finite and positive")
        if order == 2:
            if not (_finite(w) and bool((w >= 0).all())):
                raise ValueError("weights must be finite and non-negative")
            count = int((w > 0).sum())
    dev = obs.device.index if isinstance(obs, torch.Tensor) else _plan._current_device(None)
    tdev = torch.device("cuda", dev)

    def on_device(x, p0, p1):
        part = x[..., p0:p1]
        if isinstance(part, torch.Tensor):
            return part.to(tdev).contiguous()
        return torch.as_tensor(np.ascontiguousarray(part)).to(tdev)

    E = obs.shape[0]
    kp = (nmax + 1) ** 2 - nmin ** 2
    normals = torch.zeros((kp, kp), dtype=torch.float64, device=tdev)
    anm = torch.zeros((E, nmax + 1, nmax + 1), dtype=torch.float64, device=tdev)
    lpl = torch.zeros(E, dtype=torch.float64, device=tdev)
    chunk = _positions_per_chunk(nmax, order) if positions_per_chunk is None else int(positions_per_chunk)
    for p0 in range(0, P, chunk):
        p1 = min(P, p0 + chunk)
        l = on_device(obs, p0, p1)
        wc = None if w is None else on_device(w, p0, p1)
        wl = l if wc is None else l * wc
        lpl += (wl * l).sum(dim=(1, 2))
        plan = _CHUNK_PLANS[order](r[p0:p1], colat[p0:p1], lon[p0:p1], nmax, GM, R, dev)
        try:
            plan._derivative_normals(normals, nmin, frame, wc, order)
            anm += plan._derivative_adjoint(wl, frame, order)
        finally:
            plan.close()
    rhs = ravel_batch(anm, nmin).T.contiguous()
    del anm
    row_index, column_index = BlockMatrix.compute_block_index((kp, kp), int(block_size))
    matrix = BlockMatrix.from_array(normals, row_index, column_index)
    del normals
    return NormalEquations(matrix, rhs, lpl.cpu().numpy(), count)


def gridded_rms(temporal_gravityfield, epochs, kernel='ewh', base_grid=None):
    """Temporal RMS of gridded values over ``epochs`` (reference gravityfield.py:1143-1172).
    The reference synthesises epoch by epoch; here all epochs go through one batched GPU
    synthesis and the sum of squares is reduced on the device."""
    base_grid = GeographicGrid() if base_grid is None else base_grid
    fields = [temporal_gravityfield.evaluate_at(t) for t in epochs]
    if not fields:
        raise ValueError("no epochs selected")
    L = max(f.anm.shape[0] for f in fields)
    GM, R = fields[0].GM, fields[0].R
    packed = np.zeros((len(fields), L, L))
    for k, f in enumerate(fields):
        packed[k, :f.anm.shape[0], :f.anm.shape[1]] = f.anm
        if f.GM != GM or f.R != R:
            # the reference evaluates every epoch with its own constants (gravityfield.py:1165); one batched call has
            # one (GM, R), so the coefficients of such an epoch are rescaled to it: GM'/R' (R'/r)^(n+1) -> GM/R (R/r)^(n+1)
            n = np.arange(L, dtype=float)
            scale = (f.GM / GM) * (f.R / R) ** n
            packed[k] *= scale[np.maximum(np.arange(L)[:, None], np.arange(L)[None, :])]   # element (r, c) has degree max(r, c)
    values = to_grid_batch(packed, base_grid, kernel, GM, R, device_output=True)
    values = values.reshape(len(fields), -1)
    rms = torch.empty(values.shape[1], dtype=torch.float64, device=values.device)
    dev = values.device.index
    _lib.check(_lib.load().gb_temporal_rms(ctypes.c_void_p(values.data_ptr()), values.shape[0], values.shape[1],
                                           ctypes.c_void_p(rms.data_ptr()), dev, _plan._stream_handle(dev)))
    grid = base_grid.copy()
    grid.values = rms.cpu().numpy().reshape(-1)
    return grid


def grid_statistics(values, grid, mask=None):
    """Area-weighted mean, RMS and standard deviation of every epoch of a gridded batch, optionally
    inside a mask (Grid.mean / rms / std of the reference, grid.py:174-260, for [E, ...] values at once).
    values: CUDA tensor or numpy array [E, nlat, nlon] or [E, points]; mask: boolean [points] or None.
    Returns a dict of numpy arrays [E]; the grids stay on the device."""
    on_host = not isinstance(values, torch.Tensor)
    dev = _plan._current_device(None if on_host else values.device)
    v = torch.as_tensor(np.ascontiguousarray(values, dtype=float)).to(torch.device("cuda", dev)) if on_host else values.contiguous()
    v = v.reshape(v.shape[0], -1)
    if v.dtype != torch.float64 or v.shape[1] != grid.point_count:
        raise ValueError("values must be float64 with {0} points per epoch (got {1})".format(grid.point_count, tuple(v.shape)))
    # weights = area element * mask, formed on the device (the area table is cached per grid object and device)
    cache = grid.__dict__.setdefault("_gb_area_on_device", {})
    if dev not in cache:
        area = np.array(grid.area, dtype=float).reshape(-1) if grid.area is not None else np.ones(grid.point_count)
        cache[dev] = torch.as_tensor(area).to(v.device)
    wd = cache[dev]
    if mask is not None:
        mask = mask if isinstance(mask, torch.Tensor) else torch.as_tensor(np.asarray(mask, dtype=bool).reshape(-1))
        if mask.numel() != grid.point_count:
            raise ValueError("mask must have one entry per grid point")
        wd = wd * mask.reshape(-1).to(device=v.device, dtype=torch.float64)
    s0 = float(wd.sum().item())
    lib, st = _lib.load(), _plan._stream_handle(dev)
    E = v.shape[0]
    m1 = torch.empty((E, 2), dtype=torch.float64, device=v.device)
    _lib.check(lib.gb_weighted_moments(ctypes.c_void_p(v.data_ptr()), ctypes.c_void_p(wd.data_ptr()), None, E, v.shape[1],
                                       ctypes.c_void_p(m1.data_ptr()), dev, st))
    mean = m1[:, 0] / s0
    m2 = torch.empty((E, 2), dtype=torch.float64, device=v.device)
    _lib.check(lib.gb_weighted_moments(ctypes.c_void_p(v.data_ptr()), ctypes.c_void_p(wd.data_ptr()),
                                       ctypes.c_void_p(mean.contiguous().data_ptr()), E, v.shape[1],
                                       ctypes.c_void_p(m2.data_ptr()), dev, st))
    m1, m2, mean = m1.cpu().numpy(), m2.cpu().numpy(), mean.cpu().numpy()
    return {"mean": mean, "rms": np.sqrt(m1[:, 1] / s0), "std": np.sqrt(m2[:, 1] / s0)}
