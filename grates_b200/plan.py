"""Plans: the epoch-independent device tables of one (grid geometry, degree, kernel, GM, R)
combination, cached so that repeated ``to_grid`` / analysis / covariance calls pay for table
construction once.  torch is used for device memory and streams only.
"""
import ctypes
import os
import threading

import numpy as np
import torch

from . import _lib, kernel as _kernel, utilities

_cache = {}
_cache_lock = threading.Lock()
_MAX_CACHED_PLANS = 16


def _current_device(device=None):
    _lib.require_device()
    if device is None:
        return torch.cuda.current_device()
    return torch.device(device).index if not isinstance(device, int) else device


def _ptr(array):
    return array.ctypes.data_as(ctypes.c_void_p)


def _stream_handle(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _env_flag(name):
    """A switch of the CUDA library, read the way it reads it (gb_env_flag): set, non-empty, not starting with '0'."""
    return os.environ.get(name, "")[:1] not in ("", "0")


def _check_out(out, shape, device, name="out"):
    """A caller-supplied result buffer goes to the kernels as a raw pointer: it must be exactly what they write."""
    if not isinstance(out, torch.Tensor):
        raise TypeError("{0} must be a torch tensor".format(name))
    if out.dtype != torch.float64 or not out.is_cuda or out.device.index != device:
        raise ValueError("{0} must be a float64 CUDA tensor on device {1}".format(name, device))
    if tuple(out.shape) != tuple(shape) or not out.is_contiguous():
        raise ValueError("{0} must be a contiguous tensor of shape {1} (got {2})".format(name, tuple(shape), tuple(out.shape)))
    return out


def _check_out_host(out, shape, name="out"):
    if not isinstance(out, np.ndarray) or out.dtype != np.float64 or not out.flags.c_contiguous or not out.flags.writeable:
        raise ValueError("{0} must be a writeable C-contiguous float64 array".format(name))
    if tuple(out.shape) != tuple(shape):
        raise ValueError("{0} must have shape {1} (got {2})".format(name, tuple(shape), out.shape))
    return out


class PinnedArray:
    """numpy view on page-locked host memory from gb_host_alloc (full PCIe rate for *_host calls)."""

    def __init__(self, shape, dtype=np.float64):
        self._lib = _lib.load()
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        self._raw = ctypes.c_void_p()
        _lib.check(self._lib.gb_host_alloc(ctypes.byref(self._raw), self.nbytes))
        buf = (ctypes.c_char * max(self.nbytes, 1)).from_address(self._raw.value)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def free(self):
        if self._raw is not None and self._raw.value:
            self.array = None
            self._lib.gb_host_free(self._raw)
            self._raw = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class SHPlan:
    """Device-resident tables for one regular grid + kernel; wraps ``gb_plan``.

    Parameters mirror what reference ``to_grid`` derives per call (gravityfield.py:353-365):
    parallels / meridians in radians, ellipsoid (a, f), maximum degree, kernel name, GM, R.
    """

    def __init__(self, meridians, parallels, a, f, max_degree, kernel='ewh',
                 GM=3.9860044150e+14, R=6.3781363000e+06, device=None, degree_factors=None, colatitude=None):
        """degree_factors [nlat, L] / colatitude [nlat]: used instead of the kernel's factors and the ellipsoidal
        colatitudes (space-domain kernels on the unit sphere, reference kernel.py:622-658)."""
        self._lib = _lib.load()
        self.device = _current_device(device)
        self.max_degree = int(max_degree)
        self.meridians = np.ascontiguousarray(meridians, dtype=float)
        self.parallels = np.ascontiguousarray(parallels, dtype=float)
        self.a, self.f = a, f
        self.kernel, self.GM, self.R = kernel, GM, R
        self.nlat, self.nlon = self.parallels.size, self.meridians.size
        if degree_factors is None:
            colat, kn = _kernel.degree_factors(kernel, self.max_degree, self.parallels, a, f, GM, R)
        else:
            colat = utilities.colatitude(self.parallels, a, f)
            kn = np.ascontiguousarray(degree_factors, dtype=float)
            if kn.shape != (self.nlat, self.max_degree + 1):
                raise ValueError("degree_factors must have shape [{0}, {1}]".format(self.nlat, self.max_degree + 1))
        if colatitude is not None:
            colat = np.ascontiguousarray(colatitude, dtype=float)
            if colat.shape != (self.nlat,):
                raise ValueError("colatitude must have shape [{0}]".format(self.nlat))
        if not np.all(np.isfinite(kn)):
            raise ValueError("kernel '{0}' has non-finite degree factors on this grid".format(kernel))
        self.colat, self.kn = colat, kn
        cos_t = np.ascontiguousarray(np.cos(colat))
        sin_t = np.ascontiguousarray(np.sin(colat))
        cos_ml, sin_ml = utilities.trig_tables(self.max_degree, self.meridians)
        handle = ctypes.c_void_p()
        _lib.check(self._lib.gb_plan_create(ctypes.byref(handle), self.max_degree, self.nlat, self.nlon,
                                            _ptr(cos_t), _ptr(sin_t), _ptr(kn), _ptr(cos_ml), _ptr(sin_ml),
                                            self.device))
        self._handle = handle
        self._analysis_nmin = None
        self._areas_key = None
        self._lock = threading.RLock()     # one workspace per plan: host threads take turns (grates_b200.h, re-entrancy)

    # -- life cycle ---------------------------------------------------------------------
    def close(self):
        if getattr(self, "_handle", None) is not None:
            self._lib.gb_plan_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def L(self):
        return self.max_degree + 1

    @property
    def symmetric(self):
        """True if synthesis uses the four-fold longitude symmetry (see gb_plan_is_symmetric)."""
        return bool(self._lib.gb_plan_is_symmetric(self._handle)) and not _env_flag("GB_NO_SYMMETRY")

    @property
    def octant(self):
        """True if synthesis uses the eight-fold longitude symmetry (gb_plan_is_symmetric returns 2)."""
        return (self._lib.gb_plan_is_symmetric(self._handle) == 2 and not _env_flag("GB_NO_SYMMETRY")
                and not _env_flag("GB_S2_QUADRANT"))

    @property
    def folded(self):
        """True if the Legendre stage uses the equatorial symmetry of the parallels (see gb_plan_is_folded)."""
        return bool(self._lib.gb_plan_is_folded(self._handle)) and not _env_flag("GB_NO_FOLD")

    def _check_anm(self, anm):
        if anm.dim() != 3 or anm.shape[1] != self.L or anm.shape[2] != self.L:
            raise ValueError("coefficients must have shape [epochs, {0}, {0}] (got {1})".format(self.L, tuple(anm.shape)))
        if anm.dtype != torch.float64 or not anm.is_cuda or anm.device.index != self.device:
            raise ValueError("coefficients must be a float64 CUDA tensor on device {0}".format(self.device))

    # -- synthesis ----------------------------------------------------------------------
    def synthesis(self, anm, out=None, degree_weights=None, orderwise_filter=None):
        """anm: CUDA float64 tensor [E, L, L] (packed) -> CUDA tensor [E, nlat, nlon].
        degree_weights: optional [L] weights w_n of an isotropic filter (Gaussian, Butterworth),
        multiplied into the coefficients while they are packed (gb_synthesis_weighted).
        orderwise_filter: an OrderWiseFilter applied to the batch first (gb_synthesis_orderwise_filtered: its result goes
        straight into the layout the Legendre stage reads; bit-identical to filter_batch followed by synthesis).
        out: 16-byte aligned (as every torch allocation is): the kernels store pairs of doubles."""
        self._check_anm(anm)
        anm = anm.contiguous()
        E = anm.shape[0]
        if out is None:
            out = torch.empty((E, self.nlat, self.nlon), dtype=torch.float64, device=anm.device)
        else:
            _check_out(out, (E, self.nlat, self.nlon), self.device)
            if out.data_ptr() % 16:
                raise ValueError("out must be 16-byte aligned: the kernels store pairs of doubles")
        if orderwise_filter is not None:
            if degree_weights is not None:
                raise ValueError("pass either degree_weights or orderwise_filter")
            if orderwise_filter.max_degree < self.max_degree:
                raise ValueError("filter of degree {0} does not reach degree {1}".format(orderwise_filter.max_degree, self.max_degree))
            blocks = orderwise_filter._blocks_on(self.device)
            with self._lock:
                _lib.check(self._lib.gb_synthesis_orderwise_filtered(
                    self._handle, ctypes.c_void_p(blocks.data_ptr()),
                    orderwise_filter._offsets.ctypes.data_as(ctypes.c_void_p), int(orderwise_filter.max_degree),
                    ctypes.c_void_p(anm.data_ptr()), E, ctypes.c_void_p(out.data_ptr()), _stream_handle(self.device)))
            return out
        if degree_weights is not None:
            if isinstance(degree_weights, torch.Tensor):        # already on the device: no copy in the call
                w = degree_weights.to(device=anm.device, dtype=torch.float64).contiguous()
            else:
                w = torch.as_tensor(np.ascontiguousarray(degree_weights, dtype=np.float64)).to(anm.device)
            if w.numel() != self.L:
                raise ValueError("degree_weights must have {0} entries (got {1})".format(self.L, w.numel()))
            with self._lock:
                _lib.check(self._lib.gb_synthesis_weighted(self._handle, ctypes.c_void_p(anm.data_ptr()),
                                                           ctypes.c_void_p(w.data_ptr()), E,
                                                           ctypes.c_void_p(out.data_ptr()), _stream_handle(self.device)))
            return out
        with self._lock:
            _lib.check(self._lib.gb_synthesis(self._handle, ctypes.c_void_p(anm.data_ptr()), E,
                                              ctypes.c_void_p(out.data_ptr()), _stream_handle(self.device)))
        return out

    def synthesis_host(self, anm, out=None):
        """anm: numpy [E, L, L] -> numpy [E, nlat, nlon]; copies both ways inside the call."""
        anm = np.ascontiguousarray(anm, dtype=np.float64)
        if anm.ndim != 3 or anm.shape[1:] != (self.L, self.L):
            raise ValueError("coefficients must have shape [epochs, {0}, {0}] (got {1})".format(self.L, anm.shape))
        E = anm.shape[0]
        if out is None:
            out = np.empty((E, self.nlat, self.nlon))
        else:
            _check_out_host(out, (E, self.nlat, self.nlon))
        with self._lock:
            _lib.check(self._lib.gb_synthesis_host(self._handle, _ptr(anm), E, _ptr(out)))
        return out

    def legendre_table(self, scaled=False):
        """Packed Legendre table [nlat, L, L] from the on-the-fly recursion (parity hook)."""
        out = torch.empty((self.nlat, self.L, self.L), dtype=torch.float64, device=torch.device("cuda", self.device))
        _lib.check(self._lib.gb_legendre_table(self._handle, ctypes.c_void_p(out.data_ptr()), int(bool(scaled)),
                                               _stream_handle(self.device)))
        return out

    def set_profiling(self, capacity):
        """Record per-kernel CUDA events for the next ``capacity`` synthesis calls (0 = off)."""
        _lib.check(self._lib.gb_plan_set_profiling(self._handle, int(capacity)))

    def stage_times(self, max_calls=4096):
        """[calls, 3] device milliseconds of (pack, Legendre stage 1, Fourier stage 2)."""
        buf = np.zeros((max_calls, 3))
        n = ctypes.c_int(0)
        _lib.check(self._lib.gb_plan_stage_times(self._handle, buf.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                                 max_calls, ctypes.byref(n)))
        return buf[:n.value].copy()

    # -- analysis -----------------------------------------------------------------------
    def set_analysis(self, min_degree, areas):
        """Build the separable least-squares operators of reference grid.py:665-696 for the
        plan's grid (host, once) and upload them.  areas: [nlat, nlon] area weights."""
        areas = np.asarray(areas, dtype=float).reshape(self.nlat, self.nlon)
        key = (int(min_degree), hash(areas.tobytes()))
        if self._analysis_nmin == key:
            return
        if 2 * self.max_degree >= self.nlon:
            raise ValueError("analysis up to degree {0} needs more than {1} meridians (got {2})"
                             .format(self.max_degree, 2 * self.max_degree, self.nlon))
        w_lat, u_lon = separable_weights(areas)
        if _env_flag("GB_ANALYSIS_HOST_OPERATORS"):
            # cross-check: the per-order solves with numpy on the host (0.5-0.8 s at degree 180)
            lon_ops, lat_ops, offsets = analysis_operators(self, int(min_degree), w_lat, u_lon)
            with self._lock:
                _lib.check(self._lib.gb_plan_set_analysis(self._handle, int(min_degree), _ptr(lon_ops), _ptr(lat_ops),
                                                          _ptr(offsets)))
        else:
            # the latitude-side operators are built on the device (recursion, normal matrices, Cholesky solves)
            lon_ops = longitude_operators(self, u_lon)
            w = np.ascontiguousarray(w_lat, dtype=np.float64)
            with self._lock:
                _lib.check(self._lib.gb_plan_set_analysis_weights(self._handle, int(min_degree), _ptr(lon_ops), _ptr(w)))
        self._analysis_nmin = key
        self.analysis_min_degree = int(min_degree)

    def set_adjoint(self, min_degree):
        """Load the ADJOINT of the synthesis operator into the analysis slots of this plan: afterwards
        ``analysis(w)`` returns A' w (packed), A being the synthesis matrix of reference grid.py:412-443.
        Longitude operator = the trig table itself, latitude operator of order m = (kn * P_nm)'.  Used for
        functionals of gridded fields (basin means); keep such a plan separate from one used for analysis."""
        key = ("adjoint", int(min_degree))
        if self._analysis_nmin == key:
            return
        lon_ops, lat_ops, offsets = adjoint_operators(self, int(min_degree))
        with self._lock:
            _lib.check(self._lib.gb_plan_set_analysis(self._handle, int(min_degree), _ptr(lon_ops), _ptr(lat_ops),
                                                      _ptr(offsets)))
        self._analysis_nmin = key
        self.analysis_min_degree = int(min_degree)

    def analysis(self, values, out=None):
        """values: CUDA tensor [E, nlat, nlon] -> packed coefficients [E, L, L] (CUDA)."""
        if self._analysis_nmin is None:
            raise RuntimeError("call set_analysis() first")
        if values.dim() != 3 or tuple(values.shape[1:]) != (self.nlat, self.nlon):
            raise ValueError("grid values must have shape [epochs, {0}, {1}]".format(self.nlat, self.nlon))
        if values.dtype != torch.float64 or not values.is_cuda or values.device.index != self.device:
            raise ValueError("grid values must be a float64 CUDA tensor on device {0}".format(self.device))
        values = values.contiguous()
        E = values.shape[0]
        if out is None:
            out = torch.empty((E, self.L, self.L), dtype=torch.float64, device=values.device)
        else:
            _check_out(out, (E, self.L, self.L), self.device)
        with self._lock:
            _lib.check(self._lib.gb_analysis(self._handle, ctypes.c_void_p(values.data_ptr()), E,
                                             ctypes.c_void_p(out.data_ptr()), _stream_handle(self.device)))
        return out

    def synthesis_matrix(self, min_degree=0):
        """Dense synthesis operator [nlat*nlon, K'] (columns in degree-wise order) as a CUDA tensor."""
        kp = self.L ** 2 - int(min_degree) ** 2
        out = torch.zeros((self.nlat * self.nlon, kp), dtype=torch.float64, device=torch.device("cuda", self.device))
        _lib.check(self._lib.gb_synthesis_matrix(self._handle, int(min_degree), ctypes.c_void_p(out.data_ptr()),
                                                 _stream_handle(self.device)))
        return out

    def analysis_matrix(self):
        """Dense analysis operator [K', nlat*nlon] for the min_degree of set_analysis() (CUDA tensor)."""
        if self._analysis_nmin is None:
            raise RuntimeError("call set_analysis() first")
        kp = self.L ** 2 - self.analysis_min_degree ** 2
        out = torch.empty((kp, self.nlat * self.nlon), dtype=torch.float64, device=torch.device("cuda", self.device))
        _lib.check(self._lib.gb_analysis_matrix(self._handle, ctypes.c_void_p(out.data_ptr()),
                                                _stream_handle(self.device)))
        return out

    def analysis_host(self, values, out=None):
        values = np.ascontiguousarray(values, dtype=np.float64)
        if values.ndim != 3 or values.shape[1:] != (self.nlat, self.nlon):
            raise ValueError("grid values must have shape [epochs, {0}, {1}]".format(self.nlat, self.nlon))
        if self._analysis_nmin is None:
            raise RuntimeError("call set_analysis() first")
        E = values.shape[0]
        if out is None:
            out = np.empty((E, self.L, self.L))
        else:
            _check_out_host(out, (E, self.L, self.L))
        with self._lock:
            _lib.check(self._lib.gb_analysis_host(self._handle, _ptr(values), E, _ptr(out)))
        return out

    # -- covariance propagation ---------------------------------------------------------
    def covariance_propagation(self, sigma, min_degree, row0=0, nrows=None, take_sqrt=True, out=None, symmetric=None,
                               spatial_filter=None, mirrored=False):
        """sigma: CUDA tensor [K', K'] (degree-wise order, offset min_degree^2) ->
        [nrows, nlon] standard deviations (or variances) for parallels row0..row0+nrows.
        mirrored: the block is the nrows NORTHERN parallels row0.. together with their mirror images about the equator;
        the result is [2 nrows, nlon]: the northern rows, then parallels nlat-row0-nrows..nlat-row0 (GB_COV_MIRRORED: on
        equator-symmetric grids both halves share the first contraction; the way to cut row blocks for several GPUs).
        symmetric: True lets the kernels contract the order-block pairs k <= k' only (half the work);
        None (default) decides by comparing sigma with its transpose on a sample of entries.
        spatial_filter: an OrderWiseFilter, Gaussian or Butterworth instance F; the result then is the propagation
        of F sigma F' (F = spatial_filter.matrix(min_degree, max_degree)) without forming that product."""
        nrows = self.nlat - row0 if nrows is None else nrows
        kp = self.L ** 2 - min_degree ** 2
        if sigma.dim() != 2 or tuple(sigma.shape) != (kp, kp):
            raise ValueError("covariance matrix must have shape [{0}, {0}] (got {1})".format(kp, tuple(sigma.shape)))
        if sigma.dtype != torch.float64 or not sigma.is_cuda or sigma.device.index != self.device:
            raise ValueError("covariance matrix must be a float64 CUDA tensor on device {0}".format(self.device))
        sigma = sigma.contiguous()
        if symmetric is None:
            symmetric = _looks_symmetric(sigma)
        if row0 < 0 or nrows < 0 or row0 + nrows > self.nlat:
            raise ValueError("row block [{0}, {1}) is outside the grid's {2} parallels".format(row0, row0 + nrows, self.nlat))
        if mirrored and 2 * (row0 + nrows) > self.nlat:
            raise ValueError("a mirrored row block must lie north of the equator (got [{0}, {1}) of {2} parallels)".format(
                row0, row0 + nrows, self.nlat))
        nout = 2 * nrows if mirrored else nrows
        if out is None:
            out = torch.empty((nout, self.nlon), dtype=torch.float64, device=sigma.device)
        else:
            _check_out(out, (nout, self.nlon), self.device)
        flags = (1 if take_sqrt else 0) | (2 if symmetric else 0) | (4 if mirrored else 0)   # GB_COV_SQRT | _SYMMETRIC | _MIRRORED
        if spatial_filter is None:
            with self._lock:
                _lib.check(self._lib.gb_covariance_propagation(self._handle, ctypes.c_void_p(sigma.data_ptr()),
                                                               int(min_degree), int(row0), int(nrows),
                                                               ctypes.c_void_p(out.data_ptr()), flags,
                                                               _stream_handle(self.device)))
            return out
        blocks = offsets = wn = None
        nf = 0
        if hasattr(spatial_filter, "_blocks_on"):                       # order-wise blocks
            if spatial_filter.max_degree < self.max_degree:
                raise ValueError("filter of degree {0} does not reach degree {1}".format(spatial_filter.max_degree, self.max_degree))
            blocks, offsets, nf = spatial_filter._blocks_on(self.device), spatial_filter._offsets, spatial_filter.max_degree
        elif hasattr(spatial_filter, "_weights"):                       # isotropic: F = diag(w_n), every degree weighted
            wn = torch.as_tensor(np.ascontiguousarray(spatial_filter._weights(self.max_degree), dtype=np.float64)).to(sigma.device)
        else:
            raise TypeError("spatial_filter must be an OrderWiseFilter, Gaussian or Butterworth instance")
        with self._lock:
            _lib.check(self._lib.gb_covariance_propagation_filtered(
                self._handle, ctypes.c_void_p(sigma.data_ptr()), int(min_degree), int(row0), int(nrows),
                ctypes.c_void_p(out.data_ptr()), flags,
                ctypes.c_void_p(blocks.data_ptr()) if blocks is not None else None,
                offsets.ctypes.data_as(ctypes.c_void_p) if offsets is not None else None, int(nf),
                ctypes.c_void_p(wn.data_ptr()) if wn is not None else None, _stream_handle(self.device)))
        return out


_SYM_SAMPLES = {}


def _looks_symmetric(sigma, samples=16384):
    """sigma[a, b] == sigma[b, a] to 1e-13 of the largest sampled entry on a fixed pseudo-random sample of
    index pairs (a full comparison would cost as much memory traffic as the propagation itself)."""
    k = sigma.shape[0]
    key = (k, sigma.device.index)
    if key not in _SYM_SAMPLES:
        gen = torch.Generator(device="cpu").manual_seed(12345)
        a = torch.randint(0, k, (samples,), generator=gen)
        b = torch.randint(0, k, (samples,), generator=gen)
        _SYM_SAMPLES[key] = (a.to(sigma.device), b.to(sigma.device))
    a, b = _SYM_SAMPLES[key]
    u, l = sigma[a, b], sigma[b, a]
    return bool(((u - l).abs().max() <= 1e-13 * u.abs().max()).item())


def separable_weights(areas):
    """Factor areas[nlat, nlon] into w_lat[:, None] * u_lon[None, :].  The order-by-order analysis
    of the reference is only separable for rank-one area weights (all grids it constructs itself
    have them: grid.py:540, :1151, :1193); anything else is rejected, not approximated."""
    j0 = int(np.argmax(np.abs(areas).sum(axis=0)))
    i0 = int(np.argmax(np.abs(areas[:, j0])))
    if areas[i0, j0] == 0:
        raise ValueError('area elements are all zero')
    w_lat = areas[:, j0].copy()
    u_lon = areas[i0, :] / areas[i0, j0]
    if not np.allclose(w_lat[:, None] * u_lon[None, :], areas, rtol=1e-12, atol=0):
        raise ValueError('area elements are not separable into latitude and longitude factors; '
                         'the B200 analysis path does not support this grid')
    return w_lat, u_lon


def _legendre_per_order_host(nmax, m, colat):
    """Per-order Legendre columns with s = sqrt(1 - t^2), the variant the reference's analysis
    uses (utilities.py:62-115, order 0 via :138-151).  Host side: enters only the small
    plan-time least-squares operators."""
    t = np.cos(colat)
    cnt = nmax + 1 - m
    out = np.empty((t.size, cnt))
    if m == 0:
        out[:, 0] = 1
        if nmax >= 1:
            out[:, 1] = np.sqrt(3) * t
        for n in range(2, nmax + 1):
            out[:, n] = np.sqrt((2.0 * n - 1.0) * (2.0 * n + 1.0)) / n * t * out[:, n - 1] - \
                np.sqrt((2.0 * n + 1.0) / (2.0 * n - 3.0)) * (n - 1.0) / n * out[:, n - 2]
        return out
    s = np.sqrt(1 - t ** 2)
    pmm = np.sqrt(3) * s
    for n in range(2, m + 1):
        pmm = np.sqrt((2 * n + 1) / (2 * n)) * s * pmm
    out[:, 0] = pmm
    if cnt > 1:
        out[:, 1] = np.sqrt(2 * m + 3) * t * out[:, 0]
    for n in range(m + 2, nmax + 1):
        out[:, n - m] = np.sqrt((2 * n - 1) / (n - m) * (2 * n + 1) / (n + m)) * t * out[:, n - 1 - m] - \
            np.sqrt((2 * n + 1) / (2 * n - 3) * (n - m - 1) / (n - m) * (n + m - 1) / (n + m)) * out[:, n - 2 - m]
    return out


def adjoint_operators(plan, min_degree):
    """Operators that make the analysis kernels compute A' w (see SHPlan.set_adjoint)."""
    L, nlon, nlat = plan.L, plan.nlon, plan.nlat
    lam = plan.meridians
    lon_ops = np.zeros((2 * L, nlon))
    for m in range(L):
        lon_ops[2 * m] = np.cos(m * lam)
        if m > 0:
            lon_ops[2 * m + 1] = np.sin(m * lam)
    blocks, offsets = [], np.zeros(L + 1, dtype=np.int64)
    for m in range(L):
        P = (_legendre_per_order_host(plan.max_degree, m, plan.colat) * plan.kn[:, m:])[:, max(min_degree - m, 0):]
        op = np.ascontiguousarray(P.T) if P.shape[1] else np.zeros((0, nlat))
        blocks.append(op.ravel())
        offsets[m + 1] = offsets[m] + op.size
    lat_ops = np.concatenate(blocks) if offsets[-1] > 0 else np.zeros(1)
    return np.ascontiguousarray(lon_ops), np.ascontiguousarray(lat_ops), offsets


def longitude_operators(plan, u_lon):
    """lon_ops [2L][nlon] of gb_plan_set_analysis: the weighted, normalised trig rows (small: host)."""
    L, nlon = plan.L, plan.nlon
    lam = plan.meridians
    lon_ops = np.zeros((2 * L, nlon))
    for m in range(L):
        c = np.cos(m * lam)
        lon_ops[2 * m] = u_lon * c / np.sum(u_lon * c * c)
        if m > 0:
            s = np.sin(m * lam)
            lon_ops[2 * m + 1] = u_lon * s / np.sum(u_lon * s * s)
    return np.ascontiguousarray(lon_ops)


def analysis_operators(plan, min_degree, w_lat, u_lon):
    """Host construction of the separable analysis operators (see gb_plan_set_analysis)."""
    L, nlon, nlat = plan.L, plan.nlon, plan.nlat
    lon_ops = longitude_operators(plan, u_lon)
    blocks, offsets = [], np.zeros(L + 1, dtype=np.int64)
    for m in range(L):
        P = (_legendre_per_order_host(plan.max_degree, m, plan.colat) * plan.kn[:, m:])[:, max(min_degree - m, 0):]
        if P.shape[1] == 0:
            op = np.zeros((0, nlat))
        else:
            PW = (P * w_lat[:, None]).T
            op = np.linalg.solve(PW @ P, PW)
        blocks.append(np.ascontiguousarray(op).ravel())
        offsets[m + 1] = offsets[m] + op.size
    lat_ops = np.concatenate(blocks) if offsets[-1] > 0 else np.zeros(1)
    return np.ascontiguousarray(lon_ops), np.ascontiguousarray(lat_ops), offsets


class PointsPlan:
    """Device tables for an arbitrary point set (reference IrregularGrid path); wraps ``gb_points``."""

    def __init__(self, longitude, latitude, a, f, max_degree, kernel='ewh',
                 GM=3.9860044150e+14, R=6.3781363000e+06, device=None, degree_factors=None, colatitude=None):
        """degree_factors [npts, L] / colatitude [npts]: used instead of the kernel's factors and the ellipsoidal
        colatitudes (None: from ``kernel`` and the ellipsoid)."""
        self._lib = _lib.load()
        self.device = _current_device(device)
        self.max_degree = int(max_degree)
        self.longitude = np.ascontiguousarray(longitude, dtype=float)
        self.latitude = np.ascontiguousarray(latitude, dtype=float)
        if self.longitude.shape != self.latitude.shape or self.longitude.ndim != 1:
            raise ValueError("longitude and latitude must be 1-d arrays of equal length")
        self.npts = self.longitude.size
        if degree_factors is None:
            colat, kn = _kernel.degree_factors(kernel, self.max_degree, self.latitude, a, f, GM, R)
        else:
            colat = utilities.colatitude(self.latitude, a, f)
            kn = np.ascontiguousarray(degree_factors, dtype=float)
            if kn.shape != (self.npts, self.max_degree + 1):
                raise ValueError("degree_factors must have shape [{0}, {1}]".format(self.npts, self.max_degree + 1))
        if colatitude is not None:
            colat = np.ascontiguousarray(colatitude, dtype=float)
            if colat.shape != (self.npts,):
                raise ValueError("colatitude must have shape [{0}]".format(self.npts))
        if not np.all(np.isfinite(kn)):
            raise ValueError("kernel '{0}' has non-finite degree factors on this point set".format(kernel))
        self.colat, self.kn = colat, kn
        cos_t = np.ascontiguousarray(np.cos(colat))
        sin_t = np.ascontiguousarray(np.sin(colat))
        m = np.arange(self.max_degree + 1)[None, :]
        arg = self.longitude[:, None] * m                 # == m * lon, reference utilities.py:303-304
        cos_ml = np.ascontiguousarray(np.cos(arg))
        sin_ml = np.ascontiguousarray(np.sin(arg))
        handle = ctypes.c_void_p()
        _lib.check(self._lib.gb_points_create(ctypes.byref(handle), self.max_degree, self.npts, _ptr(cos_t), _ptr(sin_t),
                                              _ptr(kn), _ptr(cos_ml), _ptr(sin_ml), self.device))
        self._handle = handle

    def close(self):
        if getattr(self, "_handle", None) is not None:
            self._lib.gb_points_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def L(self):
        return self.max_degree + 1

    def synthesis(self, anm, out=None):
        """anm: CUDA float64 [E, L, L] -> CUDA tensor [E, npts]."""
        if anm.dim() != 3 or anm.shape[1] != self.L or anm.shape[2] != self.L:
            raise ValueError("coefficients must have shape [epochs, {0}, {0}] (got {1})".format(self.L, tuple(anm.shape)))
        if anm.dtype != torch.float64 or not anm.is_cuda or anm.device.index != self.device:
            raise ValueError("coefficients must be a float64 CUDA tensor on device {0}".format(self.device))
        anm = anm.contiguous()
        E = anm.shape[0]
        if out is None:
            out = torch.empty((E, self.npts), dtype=torch.float64, device=anm.device)
        else:
            _check_out(out, (E, self.npts), self.device)
        _lib.check(self._lib.gb_points_synthesis(self._handle, ctypes.c_void_p(anm.data_ptr()), E,
                                                 ctypes.c_void_p(out.data_ptr()), _stream_handle(self.device)))
        return out

    def synthesis_matrix(self, min_degree):
        """Dense synthesis operator of the point set: CUDA tensor [npts, K'] in degree-wise order."""
        k = self.L ** 2 - int(min_degree) ** 2
        out = torch.empty((self.npts, k), dtype=torch.float64, device=torch.device("cuda", self.device))
        _lib.check(self._lib.gb_points_synthesis_matrix(self._handle, int(min_degree), ctypes.c_void_p(out.data_ptr()),
                                                        _stream_handle(self.device)))
        return out

    def adjoint(self, values, out=None):
        """values: CUDA float64 [E, npts] -> CUDA tensor [E, L, L]: the transposed synthesis operator applied to
        point values (sum over points of kn * Y_nm * value, reference gravityfield.py:707-724)."""
        if values.dim() != 2 or values.shape[1] != self.npts:
            raise ValueError("values must have shape [epochs, {0}] (got {1})".format(self.npts, tuple(values.shape)))
        if values.dtype != torch.float64 or not values.is_cuda or values.device.index != self.device:
            raise ValueError("values must be a float64 CUDA tensor on device {0}".format(self.device))
        values = values.contiguous()
        E = values.shape[0]
        if out is None:
            out = torch.empty((E, self.L, self.L), dtype=torch.float64, device=values.device)
        else:
            _check_out(out, (E, self.L, self.L), self.device)
        _lib.check(self._lib.gb_points_adjoint(self._handle, ctypes.c_void_p(values.data_ptr()), E,
                                               ctypes.c_void_p(out.data_ptr()), _stream_handle(self.device)))
        return out

    def covariance_propagation(self, sigma, min_degree, take_sqrt=True, symmetric=None):
        """sigma: CUDA tensor [K', K'] in degree-wise order -> [npts] standard deviations / variances.
        symmetric: contract only the lower triangle of sigma (half the flops); None decides on sampled entries."""
        kp = self.L ** 2 - min_degree ** 2
        if sigma.dim() != 2 or tuple(sigma.shape) != (kp, kp):
            raise ValueError("covariance matrix must have shape [{0}, {0}] (got {1})".format(kp, tuple(sigma.shape)))
        if sigma.dtype != torch.float64 or not sigma.is_cuda or sigma.device.index != self.device:
            raise ValueError("covariance matrix must be a float64 CUDA tensor on device {0}".format(self.device))
        sigma = sigma.contiguous()
        if symmetric is None:
            symmetric = _looks_symmetric(sigma)
        out = torch.empty((self.npts,), dtype=torch.float64, device=sigma.device)
        flags = (1 if take_sqrt else 0) | (2 if symmetric else 0)      # GB_COV_SQRT | GB_COV_SYMMETRIC
        _lib.check(self._lib.gb_points_covariance(self._handle, ctypes.c_void_p(sigma.data_ptr()), int(min_degree),
                                                  ctypes.c_void_p(out.data_ptr()), flags,
                                                  _stream_handle(self.device)))
        return out

    def gradient_covariance(self, sigma, min_degree, frame='cartesian', full=False):
        """Covariance of grad V at the points of a gradient point plan (get_gradient_points_plan: degree N + 1 for a
        degree-N field): sigma CUDA tensor [K', K'], K' = (N + 1)^2 - min_degree^2 in degree-wise order, contracted as
        its symmetric part (Sigma + Sigma') / 2.  frame 'cartesian' (x, y, z) or 'local' (east, north, up).  Returns a
        CUDA tensor [npts, 3, 3] of covariances in (m/s^2)^2 with full=True, else [3, npts] standard deviations in m/s^2
        (gb_points_gradient_covariance)."""
        if frame not in ('cartesian', 'local'):
            raise ValueError("frame must be 'cartesian' or 'local' (got {0!r})".format(frame))
        if not hasattr(self, "frame"):
            raise ValueError("gradient_covariance needs a gradient point plan (get_gradient_points_plan)")
        nmax = self.max_degree - 1
        if not 0 <= min_degree <= nmax:
            raise ValueError("min_degree={0} outside [0, {1}]".format(min_degree, nmax))
        kp = (nmax + 1) ** 2 - min_degree ** 2
        if sigma.dim() != 2 or tuple(sigma.shape) != (kp, kp):
            raise ValueError("covariance matrix must have shape [{0}, {0}] (got {1})".format(kp, tuple(sigma.shape)))
        if sigma.dtype != torch.float64 or not sigma.is_cuda or sigma.device.index != self.device:
            raise ValueError("covariance matrix must be a float64 CUDA tensor on device {0}".format(self.device))
        sigma = sigma.contiguous()
        shape = (self.npts, 3, 3) if full else (3, self.npts)
        out = torch.empty(shape, dtype=torch.float64, device=sigma.device)
        fr = ctypes.c_void_p(self.frame.data_ptr()) if frame == 'local' else None
        _lib.check(self._lib.gb_points_gradient_covariance(self._handle, ctypes.c_void_p(sigma.data_ptr()),
                                                           int(min_degree), fr, ctypes.c_void_p(out.data_ptr()),
                                                           0 if full else 1, _stream_handle(self.device)))   # GB_COV_SQRT
        return out

    def _gradient_field_degree(self, frame, min_degree, name):
        if frame not in ('cartesian', 'local'):
            raise ValueError("frame must be 'cartesian' or 'local' (got {0!r})".format(frame))
        if not hasattr(self, "frame"):
            raise ValueError("{0} needs a gradient point plan (get_gradient_points_plan)".format(name))
        nmax = self.max_degree - 1
        if not 0 <= min_degree <= nmax:
            raise ValueError("min_degree={0} outside [0, {1}]".format(min_degree, nmax))
        return nmax

    def gradient_normals(self, normals, min_degree, frame='cartesian', weights=None):
        """Adds the normal equations sum_p J~_p' W_p J~_p of acceleration observations at the points of a gradient point
        plan to ``normals``, a CUDA float64 tensor [K', K'] (K' = (N + 1)^2 - min_degree^2, degree-wise; zeroed by the
        caller for a fresh matrix), and returns it with both triangles holding the sum.  J~_p: the Jacobian of grad V in
        ``frame`` ('cartesian' or 'local'); weights: CUDA float64 tensor [3, npts] of positive weights (inverse variances)
        or None for 1 (gb_points_gradient_normals)."""
        nmax = self._gradient_field_degree(frame, min_degree, "gradient_normals")
        kp = (nmax + 1) ** 2 - min_degree ** 2
        if normals.dim() != 2 or tuple(normals.shape) != (kp, kp) or not normals.is_contiguous():
            raise ValueError("normal matrix must be a contiguous tensor of shape [{0}, {0}] (got {1})".format(
                kp, tuple(normals.shape)))
        if normals.dtype != torch.float64 or not normals.is_cuda or normals.device.index != self.device:
            raise ValueError("normal matrix must be a float64 CUDA tensor on device {0}".format(self.device))
        w = None
        if weights is not None:
            if tuple(weights.shape) != (3, self.npts):
                raise ValueError("weights must have shape [3, {0}] (got {1})".format(self.npts, tuple(weights.shape)))
            if weights.dtype != torch.float64 or not weights.is_cuda or weights.device.index != self.device:
                raise ValueError("weights must be a float64 CUDA tensor on device {0}".format(self.device))
            weights = weights.contiguous()
            w = ctypes.c_void_p(weights.data_ptr())
        fr = ctypes.c_void_p(self.frame.data_ptr()) if frame == 'local' else None
        _lib.check(self._lib.gb_points_gradient_normals(self._handle, int(min_degree), w, fr,
                                                        ctypes.c_void_p(normals.data_ptr()), _stream_handle(self.device)))
        return normals

    def gradient_adjoint(self, values, frame='cartesian'):
        """Transpose of the acceleration at the points of a gradient point plan: values CUDA float64 [E, 3, npts] in
        ``frame`` -> CUDA tensor [E, N + 1, N + 1] packed, sum_p J_p' Q_p' v_p: Q' for 'local' (gb_rotate_from_local), the
        adjoint synthesis of the 3E component sets (``adjoint``) and T' (gb_gradient_coefficients_adjoint)."""
        nmax = self._gradient_field_degree(frame, 0, "gradient_adjoint")
        if values.dim() != 3 or values.shape[1] != 3 or values.shape[2] != self.npts:
            raise ValueError("values must have shape [sets, 3, {0}] (got {1})".format(self.npts, tuple(values.shape)))
        if values.dtype != torch.float64 or not values.is_cuda or values.device.index != self.device:
            raise ValueError("values must be a float64 CUDA tensor on device {0}".format(self.device))
        E = values.shape[0]
        st = _stream_handle(self.device)
        if frame == 'local':
            values = values.clone(memory_format=torch.contiguous_format)
            _lib.check(self._lib.gb_rotate_from_local(ctypes.c_void_p(values.data_ptr()),
                                                      ctypes.c_void_p(self.frame.data_ptr()), E, self.npts, self.device,
                                                      st))
        g = self.adjoint(values.contiguous().view(3 * E, self.npts))
        out = torch.empty((E, nmax + 1, nmax + 1), dtype=torch.float64, device=values.device)
        _lib.check(self._lib.gb_gradient_coefficients_adjoint(ctypes.c_void_p(g.data_ptr()), E, nmax,
                                                              ctypes.c_void_p(out.data_ptr()), self.device, st))
        return out


def get_points_plan(grid, max_degree, kernel='ewh', GM=3.9860044150e+14, R=6.3781363000e+06, device=None):
    """Cached PointsPlan for a grid object exposing .longitude/.latitude/.semimajor_axis/.flattening."""
    dev = _current_device(device)
    lon = np.asarray(grid.longitude, dtype=float)
    lat = np.asarray(grid.latitude, dtype=float)
    key = ("points", lon.tobytes(), lat.tobytes(), float(grid.semimajor_axis), float(grid.flattening),
           int(max_degree), kernel.lower(), float(GM), float(R), dev)
    return _cached(key, lambda: PointsPlan(lon, lat, grid.semimajor_axis, grid.flattening, max_degree, kernel, GM, R, dev))


def is_regular(grid):
    return hasattr(grid, "parallels") and hasattr(grid, "meridians")


def get_plan(grid, max_degree, kernel='ewh', GM=3.9860044150e+14, R=6.3781363000e+06, device=None, variant=''):
    """Cached plan for a regular grid object exposing .meridians/.parallels/.semimajor_axis/.flattening.
    variant: extra cache key for plans whose analysis slots hold other operators (the adjoint)."""
    try:
        meridians, parallels = grid.meridians, grid.parallels
    except AttributeError:
        raise NotImplementedError("this call needs a regular grid (meridians x parallels); use the point-set "
                                  "entry points for irregular grids -- there is no CPU fallback") from None
    dev = _current_device(device)
    key = (np.asarray(meridians, dtype=float).tobytes(), np.asarray(parallels, dtype=float).tobytes(),
           float(grid.semimajor_axis), float(grid.flattening), int(max_degree), kernel.lower(), float(GM), float(R), dev,
           variant)
    return _cached(key, lambda: SHPlan(meridians, parallels, grid.semimajor_axis, grid.flattening, max_degree, kernel, GM,
                                       R, dev))


def _cached(key, make):
    with _cache_lock:
        plan = _cache.get(key)
        if plan is None:
            plan = make()
            if len(_cache) >= _MAX_CACHED_PLANS:
                _cache.pop(next(iter(_cache)))       # destroyed by __del__ once no caller holds it any more
            _cache[key] = plan
        return plan


def _derivative_degree_factors(radius, max_degree, order, GM, R):
    """kn[p, n] = GM/R^(order+1) (R/r_p)^(n+1), n = 0..max_degree + order; columns 0..order-1 are zero (those degrees of
    the transformed coefficients are)."""
    kn = np.power((R / np.asarray(radius, dtype=float))[:, None], np.arange(max_degree + order + 1, dtype=int) + 1) * (
        GM / R ** (order + 1))
    kn[:, :order] = 0.0
    return kn


def gradient_degree_factors(radius, max_degree, GM, R):
    """Degree factors kn'[p, n'] = GM/R^2 (R/r_p)^(n'+1), n' = 0..max_degree + 1, of the syntheses that turn the output of
    gb_gradient_coefficients into the components of grad V; column 0 is zero (degree 0 of those coefficients is)."""
    return _derivative_degree_factors(radius, max_degree, 1, GM, R)


def gravity_gradient_degree_factors(radius, max_degree, GM, R):
    """Degree factors kn''[p, n''] = GM/R^3 (R/r_p)^(n''+1), n'' = 0..max_degree + 2, of the syntheses that turn the output
    of gb_gravity_gradient_coefficients into the components of the gravity gradient tensor; columns 0 and 1 are zero."""
    return _derivative_degree_factors(radius, max_degree, 2, GM, R)


def _frame_table(colat, lon, device):
    """[4, P] device table (cos theta, sin theta, cos lon, sin lon) that gb_rotate_to_local reads."""
    table = np.stack((np.cos(colat), np.sin(colat), np.cos(lon), np.sin(lon)))
    return torch.as_tensor(np.ascontiguousarray(table)).to(torch.device("cuda", device))


# order of the derivative -> (name, cache variant of the grid plan, of the point plan)
_DERIVATIVES = {1: ("gradient", "gradient", "gradient points"),
                2: ("gravity gradient", "gravity gradient", "gravity gradient points")}


def _derivative_plan(grid, max_degree, order, GM, R, device):
    dev = _current_device(device)
    meridians = np.asarray(grid.meridians, dtype=float)
    parallels = np.asarray(grid.parallels, dtype=float)
    a, f = float(grid.semimajor_axis), float(grid.flattening)
    name, variant, _ = _DERIVATIVES[order]
    key = (meridians.tobytes(), parallels.tobytes(), a, f, int(max_degree), float(GM), float(R), dev, variant)

    def make():
        kn = _derivative_degree_factors(utilities.geocentric_radius(parallels, a, f), int(max_degree), order, GM, R)
        plan = SHPlan(meridians, parallels, a, f, int(max_degree) + order, name, GM, R, dev, degree_factors=kn)
        nlat, nlon = plan.nlat, plan.nlon
        plan.frame = _frame_table(np.repeat(plan.colat, nlon), np.tile(meridians, nlat), dev)
        return plan
    return _cached(key, make)


def get_gradient_plan(grid, max_degree, GM=3.9860044150e+14, R=6.3781363000e+06, device=None):
    """Cached SHPlan at degree max_degree + 1 for the gradient of degree-max_degree coefficients on a regular grid:
    the grid's geocentric colatitudes, the degree factors of gradient_degree_factors at the geocentric radius of each
    parallel, and ``plan.frame`` [4, nlat * nlon], the per-point table of the rotation to (east, north, up).  Its cache
    key carries a 'gradient' variant: it is never mistaken for a potential plan of the same grid and degree."""
    return _derivative_plan(grid, max_degree, 1, GM, R, device)


def get_gravity_gradient_plan(grid, max_degree, GM=3.9860044150e+14, R=6.3781363000e+06, device=None):
    """Cached SHPlan at degree max_degree + 2 for the gravity gradient tensor of degree-max_degree coefficients on a
    regular grid: as get_gradient_plan, with the degree factors of gravity_gradient_degree_factors.  Its cache key
    carries its own variant: it is never mistaken for the gradient plan of degree max_degree + 1, which has the same
    degree and other factors."""
    return _derivative_plan(grid, max_degree, 2, GM, R, device)


def _derivative_points_plan(radius, colat, lon, max_degree, order, GM, R, device, cached):
    dev = _current_device(device)
    radius, colat, lon = (np.ascontiguousarray(v, dtype=float) for v in (radius, colat, lon))
    name, _, variant = _DERIVATIVES[order]

    def make():
        kn = _derivative_degree_factors(radius, int(max_degree), order, GM, R)
        plan = PointsPlan(lon, 0.5 * np.pi - colat, utilities.A_GRS80, utilities.F_GRS80, int(max_degree) + order, name,
                          GM, R, dev, degree_factors=kn, colatitude=colat)
        plan.frame = _frame_table(colat, lon, dev)
        return plan
    if not cached:
        return make()
    key = (variant, radius.tobytes(), colat.tobytes(), lon.tobytes(), int(max_degree), float(GM), float(R), dev)
    return _cached(key, make)


def get_gradient_points_plan(radius, colat, lon, max_degree, GM=3.9860044150e+14, R=6.3781363000e+06, device=None):
    """Cached PointsPlan at degree max_degree + 1 for the gradient at points of geocentric radius / colatitude /
    longitude (any radius: on the ellipsoid for an IrregularGrid, anywhere for Cartesian positions), with ``plan.frame``
    [4, P] as for get_gradient_plan."""
    return _derivative_points_plan(radius, colat, lon, max_degree, 1, GM, R, device, True)


def gradient_points_plan(radius, colat, lon, max_degree, GM=3.9860044150e+14, R=6.3781363000e+06, device=None):
    """The PointsPlan of get_gradient_points_plan, not cached: the caller closes it (long position arrays in chunks)."""
    return _derivative_points_plan(radius, colat, lon, max_degree, 1, GM, R, device, False)


def get_gravity_gradient_points_plan(radius, colat, lon, max_degree, GM=3.9860044150e+14, R=6.3781363000e+06,
                                     device=None):
    """Cached PointsPlan at degree max_degree + 2 for the gravity gradient tensor at points, as get_gradient_points_plan
    with the degree factors of gravity_gradient_degree_factors and its own cache variant."""
    return _derivative_points_plan(radius, colat, lon, max_degree, 2, GM, R, device, True)


def clear_plan_cache():
    """Destroy the cached plans and hand the library's pooled scratch memory back to the driver (gb_trim)."""
    with _cache_lock:
        devices = {plan.device for plan in _cache.values()}
        for plan in _cache.values():
            plan.close()
        _cache.clear()
    lib = _lib.load()
    for dev in devices:
        _lib.check(lib.gb_trim(int(dev)))


def legendre_table_for_colatitudes(max_degree, colat, device=None):
    """utilities.legendre_functions for arbitrary colatitudes via the device recursion."""
    lib = _lib.load()
    dev = _current_device(device)
    L = max_degree + 1
    cos_t = np.ascontiguousarray(np.cos(colat))
    sin_t = np.ascontiguousarray(np.sin(colat))
    kn = np.ones((colat.size, L))
    dummy = np.ones((L, 1))
    handle = ctypes.c_void_p()
    _lib.check(lib.gb_plan_create(ctypes.byref(handle), max_degree, colat.size, 1, _ptr(cos_t), _ptr(sin_t), _ptr(kn),
                                  _ptr(dummy), _ptr(dummy), dev))
    try:
        out = torch.empty((colat.size, L, L), dtype=torch.float64, device=torch.device("cuda", dev))
        _lib.check(lib.gb_legendre_table(handle, ctypes.c_void_p(out.data_ptr()), 0, _stream_handle(dev)))
        result = out.cpu().numpy()
    finally:
        lib.gb_plan_destroy(handle)
    return result
