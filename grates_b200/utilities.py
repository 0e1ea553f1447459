"""Host-side helpers mirroring grates.utilities for the spherical-harmonic hot path.

Only small, epoch-independent quantities are computed here (ellipsoid geometry, index
permutations, trigonometric tables).  The Legendre functions are evaluated on the GPU:
``legendre_functions`` below is a thin wrapper around the CUDA recursion kernel.
"""
import numpy as np

A_GRS80 = 6378137.0
F_GRS80 = 298.2572221010 ** -1


def geocentric_radius(latitude, a=A_GRS80, f=F_GRS80):
    """Geocentric radius of points on the ellipsoid (reference utilities.py:414-435)."""
    e2 = f * (2 - f)
    sin_lat = np.sin(latitude)
    nu = a / np.sqrt(1 - e2 * sin_lat ** 2)
    return nu * np.sqrt(np.cos(latitude) ** 2 + (1 - e2) ** 2 * sin_lat ** 2)


def colatitude(latitude, a=A_GRS80, f=F_GRS80):
    """Geocentric colatitude of points on the ellipsoid (reference utilities.py:438-459)."""
    e2 = f * (2 - f)
    nu = a / np.sqrt(1 - e2 * np.sin(latitude) ** 2)
    return np.arccos(nu * (1 - e2) * np.sin(latitude) / geocentric_radius(latitude, a, f))


def cartesian_to_spherical(positions):
    """Earth-fixed Cartesian positions [P, 3] in metres -> geocentric (radius, colatitude, longitude), each [P]:
    r = |x|, theta = atan2(sqrt(x^2 + y^2), z), lon = atan2(y, x), with lon = 0 on the polar axis.
    Non-finite positions and the origin (r = 0) raise ValueError."""
    x = np.asarray(positions, dtype=float)
    if x.ndim != 2 or x.shape[1] != 3:
        raise ValueError("positions must have shape [points, 3] (got {0})".format(x.shape))
    if not np.all(np.isfinite(x)):
        raise ValueError("positions must be finite")
    rho = np.sqrt(x[:, 0] ** 2 + x[:, 1] ** 2)
    r = np.sqrt(x[:, 0] ** 2 + x[:, 1] ** 2 + x[:, 2] ** 2)
    if np.any(r == 0):
        raise ValueError("positions must not be the origin (r = 0)")
    lon = np.where(rho > 0, np.arctan2(x[:, 1], x[:, 0]), 0.0)
    return r, np.arctan2(rho, x[:, 2]), lon


_INDEX_CACHE = {}


def degreewise_index(min_degree, max_degree):
    """Row / column indices into the packed [L, L] array, in degree-wise vector order
    (per degree: C_n0, then C_nm, S_nm for m = 1..n; reference utilities.py:336-343)."""
    key = (min_degree, max_degree)
    if key not in _INDEX_CACHE:
        rows, cols = [], []
        for n in range(min_degree, max_degree + 1):
            m = np.arange(1, n + 1)
            r = np.empty(2 * n + 1, dtype=np.int64)
            c = np.empty(2 * n + 1, dtype=np.int64)
            r[0], c[0] = n, 0
            r[1::2], c[1::2] = n, m
            r[2::2], c[2::2] = m - 1, n
            rows.append(r)
            cols.append(c)
        if rows:
            _INDEX_CACHE[key] = (np.concatenate(rows), np.concatenate(cols))
        else:
            _INDEX_CACHE[key] = (np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64))
    return _INDEX_CACHE[key]


def ravel_coefficients(array, min_degree=0, max_degree=None):
    """Packed [L, L] or [k, L, L] array -> degree-wise vector(s) (reference utilities.py:310-360)."""
    array = np.asarray(array)
    if array.ndim not in (2, 3):
        raise ValueError('Only 2d or 3d spherical harmonic arrays can be raveled.')
    if max_degree is None:
        max_degree = array.shape[-1] - 1
    count = (max_degree + 1) ** 2 - min_degree ** 2
    rows, cols = degreewise_index(min_degree, min(array.shape[-1] - 1, max_degree))
    out = np.zeros(array.shape[:-2] + (count,), dtype=array.dtype)
    out[..., :rows.size] = array[..., rows, cols]
    return out


def unravel_coefficients(vector, min_degree=0, max_degree=None):
    """Degree-wise vector(s) -> packed array(s) (reference utilities.py:363-411)."""
    vector = np.asarray(vector)
    if vector.ndim not in (1, 2):
        raise ValueError('Only 1d or 2d spherical harmonic vectors can be unraveled.')
    if max_degree is None:
        max_degree = int(np.sqrt(vector.shape[-1] + min_degree * min_degree) - 1)
    rows, cols = degreewise_index(min_degree, max_degree)
    out = np.zeros(vector.shape[:-1] + (max_degree + 1, max_degree + 1), dtype=vector.dtype)
    out[..., rows, cols] = vector[..., :rows.size]
    return out


def trigonometric_functions(max_degree, lon):
    """Packed cos(m lon) / sin(m lon) table [points, L, L] (reference utilities.py:249-275)."""
    lam = np.atleast_1d(lon)
    L = max_degree + 1
    cs = np.empty((lam.size, L, L))
    cs[:, :, 0] = 1
    for m in range(1, L):
        cs[:, m:, m] = np.cos(m * lam)[:, None]
        cs[:, m - 1, m:] = np.sin(m * lam)[:, None]
    return cs


def trig_tables(max_degree, lon):
    """cos(m lon_j), sin(m lon_j) as two [L, nlon] tables -- the compact form the CUDA plan takes.
    Each entry is evaluated as np.cos(m * lon) exactly like reference utilities.py:271-273."""
    lam = np.atleast_1d(np.asarray(lon, dtype=float))
    m = np.arange(max_degree + 1)[:, None]
    arg = m * lam[None, :]
    return np.ascontiguousarray(np.cos(arg)), np.ascontiguousarray(np.sin(arg))


def legendre_functions(max_degree, colat, device=None):
    """Fully normalised associated Legendre functions in the reference's packed layout
    (reference utilities.py:13-59), evaluated by the CUDA recursion kernel.  Returns a numpy
    array [points, L, L] bit-identical to the reference table."""
    from .plan import legendre_table_for_colatitudes
    return legendre_table_for_colatitudes(max_degree, np.atleast_1d(np.asarray(colat, dtype=float)), device)
