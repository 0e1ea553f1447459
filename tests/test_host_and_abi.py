"""CPU-side tests: the C-ABI library loads and exports every declared symbol, host logic of the
Python mirror agrees with the golden reference outputs, nothing computes without a GPU."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import ROOT, maxnorm_err

gb = pytest.importorskip("grates_b200")


def test_library_exports_every_header_symbol():
    header = open(os.path.join(ROOT, "include", "grates_b200.h")).read()
    declared = set(re.findall(r"\b(gb_[a-z0-9_]+)\s*\(", header))
    declared.discard("gb_plan")
    assert len(declared) >= 18
    lib = gb._lib.load()
    for name in sorted(declared):
        assert hasattr(lib, name), name
    assert declared == set(gb._lib.SIGNATURES), declared ^ set(gb._lib.SIGNATURES)
    assert lib.gb_version() >= 100
    raw = ctypes.CDLL(gb._lib.library_path())
    for name in declared:
        getattr(raw, name)


def test_header_is_plain_c_and_links_from_c(tmp_path):
    """The boundary is a C ABI, not a C++ or Python one: a C99 translation unit includes the header, takes the address of
    every declared entry point, links against the shared library and runs -- what a cgo / JNI / FFI binding would do.
    No compute call is made (there is no GPU here): gb_version answers, a NULL plan is refused with an error message."""
    import shutil
    import subprocess
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    header = open(os.path.join(ROOT, "include", "grates_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(gb_[a-z0-9_]+)\s*\(", header)) - {"gb_plan"})
    src = tmp_path / "abi.c"
    src.write_text(
        '#include <stdio.h>\n#include "grates_b200.h"\n'
        "typedef void (*fn)(void);\n"
        "static fn table[] = {" + ", ".join("(fn)%s" % n for n in declared) + "};\n"
        "int main(void) {\n"
        "  unsigned i, n = 0;\n"
        "  for (i = 0; i < sizeof table / sizeof table[0]; ++i) n += table[i] != 0;\n"
        "  int rc = gb_synthesis(0, 0, 1, 0, 0);\n"
        '  printf("%d %u %d %s\\n", gb_version(), n, rc, gb_last_error());\n'
        "  return rc == GB_OK;\n"
        "}\n")
    exe = tmp_path / "abi"
    libdir = os.path.dirname(gb._lib.library_path())
    gb._lib.load()                                                         # builds the library when it is missing
    subprocess.run([cc, "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                    "-L", libdir, "-lgrates_b200", "-Wl,-rpath," + libdir], check=True, capture_output=True, text=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split(None, 3)
    assert int(out[0]) == gb._lib.GB_VERSION and int(out[1]) == len(declared)
    assert int(out[2]) != 0 and "plan is NULL" in out[3]


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(RuntimeError):
        gb.PotentialCoefficients(max_degree=4).to_grid(gb.GeographicGrid(30.0, 30.0))
    g = gb.GeographicGrid(30.0, 30.0)
    g.values = np.zeros(g.point_count)
    with pytest.raises(RuntimeError):
        g.to_potential_coefficients(0, 2)
    with pytest.raises(RuntimeError):
        gb.OrderWiseFilter([np.eye(2), np.eye(1), np.eye(1)]).filter(gb.PotentialCoefficients(max_degree=1))


def test_product_does_not_import_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "grates_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text and "sh_oracle" not in text, f


def test_host_grids_match_reference(golden):
    g = golden("grids")
    geo = gb.GeographicGrid(2.0, 4.0)
    np.testing.assert_array_equal(geo.meridians, g["geo_meridians"])
    np.testing.assert_array_equal(geo.parallels, g["geo_parallels"])
    np.testing.assert_array_equal(geo.area, g["geo_area"])
    ga = gb.GaussGrid(14)
    np.testing.assert_array_equal(ga.parallels, g["gauss_parallels"])
    np.testing.assert_array_equal(ga.area, g["gauss_area"])
    rg = gb.RegularGrid(g["reg_meridians"], g["reg_parallels"])
    np.testing.assert_array_equal(rg.area, g["reg_area"])
    c = geo.copy()
    assert type(c) is gb.GeographicGrid and c.value_array is None and c.point_count == 45 * 180
    with pytest.raises(ValueError):
        c.values = np.zeros(3)
    with pytest.raises(ValueError):
        c.values = np.zeros((2, 2))
    c.values = np.arange(c.point_count, dtype=float)
    assert c.value_array.shape == (45, 180) and c.copy().values[7] == 7.0
    assert c.mean() == pytest.approx(np.sum(c.area * c.values) / np.sum(c.area))
    np.testing.assert_array_equal(c.longitude[:180], c.meridians)
    np.testing.assert_array_equal(c.latitude[:180], np.full(180, c.parallels[0]))


@pytest.mark.parametrize("name", ["ewh", "obp", "potential", "geoid", "surface_density", "anomaly", "deformation", "uplift"])
def test_host_kernel_factors_match_reference(golden, name):
    g = golden("kernels")
    k = gb.get_kernel(name)
    np.testing.assert_allclose(k.coefficients(0, 24, g["r"], g["colat"]), g["coeff_" + name], rtol=1e-14, atol=0)
    np.testing.assert_allclose(k.inverse_coefficients(0, 24, g["r"], g["colat"]), g["inv_" + name], rtol=1e-14, atol=0)
    _, kn = gb.kernel.degree_factors(name, 24, g["lat"], 6378137.0, 298.2572221010 ** -1, 3.9860044150e+14, 6.3781363000e+06)
    np.testing.assert_allclose(kn, g["kn_" + name], rtol=1e-14, atol=0)
    if name in ("ewh", "potential", "surface_density", "anomaly"):
        np.testing.assert_array_equal(kn, g["kn_" + name])


def test_host_kernel_errors_and_normal_gravity(golden):
    g = golden("kernels")
    with pytest.raises(ValueError):
        gb.get_kernel("nope")
    with pytest.raises(ValueError):
        gb.get_kernel("ewh").coefficients(0, 3, np.ones(3), np.ones(4))
    np.testing.assert_allclose(gb.kernel.normal_gravity(g["r"], g["colat"]), g["normal_gravity"], rtol=1e-14)
    np.testing.assert_allclose(gb.kernel.normal_gravity(6378137.0, np.pi / 2), 9.7803267715, rtol=1e-11)
    assert gb.get_kernel("EWH").__class__ is gb.kernel.WaterHeight
    with pytest.raises(ValueError):
        gb.kernel.load_love_numbers("xx")


def test_host_utilities_match_reference(golden):
    g = golden("l1_numerics")
    u = gb.utilities
    np.testing.assert_array_equal(u.ravel_coefficients(g["ravel_in"], 0, 6), g["ravel_0_6"])
    np.testing.assert_array_equal(u.ravel_coefficients(g["ravel_in"], 2, 6), g["ravel_2_6"])
    np.testing.assert_array_equal(u.ravel_coefficients(g["ravel_in"][0], 2, 4), g["ravel_2_4"])
    np.testing.assert_array_equal(u.unravel_coefficients(g["unravel_in"], 2, 6), g["unravel_2_6"])
    np.testing.assert_array_equal(u.geocentric_radius(g["lat"]), g["geocentric_radius"])
    np.testing.assert_array_equal(u.colatitude(g["lat"]), g["colatitude"])
    np.testing.assert_array_equal(u.trigonometric_functions(12, g["lon"]), g["trig_12"])
    c, s = u.trig_tables(12, g["lon"])
    np.testing.assert_array_equal(c[5], g["trig_12"][:, 7, 5])
    np.testing.assert_array_equal(s[5], g["trig_12"][:, 4, 9])
    with pytest.raises(ValueError):
        u.ravel_coefficients(np.zeros(4))


def test_potential_coefficients_container(golden):
    g = golden("filters")
    pc = gb.PotentialCoefficients(max_degree=4)
    assert pc.anm.shape == (5, 5) and pc.max_degree == 4 and pc.epoch is None
    pc.anm = g["ts_anm_sorted"][0].copy()
    np.testing.assert_array_equal(pc.values, g["ts_array"][0])
    q = pc.copy()
    q.values = pc.values * 2
    np.testing.assert_array_equal(q.anm, pc.anm * 2)
    np.testing.assert_allclose((pc + q).anm, pc.anm * 3, rtol=1e-15)
    np.testing.assert_allclose((q - pc).anm, pc.anm, rtol=1e-15)
    np.testing.assert_array_equal((pc * 2).anm, q.anm)
    with pytest.raises(TypeError):
        pc + 1
    with pytest.raises(TypeError):
        pc * "a"
    rows, cols = gb.gravityfield.degree_indices(3)
    assert list(rows) == [3, 3, 3, 3, 0, 1, 2] and list(cols) == [0, 1, 2, 3, 3, 3, 3]
    rows, cols = gb.gravityfield.order_indices(3, 2)
    assert list(rows) == [2, 3, 1, 1] and list(cols) == [2, 2, 2, 3]
    import datetime
    data = []
    for e in range(3):
        p = gb.PotentialCoefficients()
        p.anm = g["ts_anm_sorted"][e].copy()
        p.epoch = datetime.datetime(2002, 4, 15) + datetime.timedelta(days=30.4375 * e)
        data.append(p)
    ts = gb.TimeSeries(data[::-1])
    np.testing.assert_array_equal(ts.to_array(), g["ts_array"])
    assert len(ts) == 3 and ts[0].epoch < ts[1].epoch
    mid = ts.interpolate_to(data[0].epoch + (data[1].epoch - data[0].epoch) / 2)
    np.testing.assert_allclose(mid.anm, 0.5 * (data[0].anm + data[1].anm), rtol=1e-14, atol=1e-30)
    with pytest.raises(ValueError):
        ts.interpolate_to(datetime.datetime(1990, 1, 1))
    bad = gb.PotentialCoefficients()
    with pytest.raises(ValueError):
        gb.TimeSeries([bad])


def test_orderwise_filter_host_side(golden):
    g = golden("filters")
    blocks = [g["block_%02d" % i] for i in range(25)]
    flt = gb.OrderWiseFilter(blocks)
    assert flt.max_degree == 12
    np.testing.assert_array_equal(flt.matrix(2, 9), g["matrix_2_9"])
    with pytest.raises(ValueError):
        gb.OrderWiseFilter(blocks[:-1])
    with pytest.raises(TypeError):
        flt.filter("x")
    big = gb.PotentialCoefficients(max_degree=13)
    with pytest.raises(ValueError):
        flt.filter(big)


def test_analysis_operator_host_construction(golden):
    """The separable operators reproduce the reference's solve(A'WA, A'W) per order."""
    from oracle import sh_oracle as orc
    from grates_b200 import plan as gplan
    og = orc.geographic_grid(30.0, 30.0)

    class FakePlan:
        pass
    fp = FakePlan()
    fp.max_degree, fp.L, fp.nlat, fp.nlon = 4, 5, 6, 12
    fp.meridians = og.meridians
    fp.colat, fp.kn = orc.kn_table("ewh", 4, og.parallels)
    w, u = gplan.separable_weights(og.areas)
    lon_ops, lat_ops, off = gplan.analysis_operators(fp, 0, w, u)
    g = golden("analysis")
    ref = g["analysis_matrix_0_4"]                       # [25, 72] rows in degree-wise order
    rows, cols = gb.utilities.degreewise_index(0, 4)
    full = np.zeros((25, 72))
    for a, (r, c) in enumerate(zip(rows, cols)):
        m, n, cs = (c, r, 0) if c <= r else (r + 1, c, 1)
        op = lat_ops[off[m]:off[m + 1]].reshape(-1, 6)
        full[a] = np.outer(op[n - m], lon_ops[2 * m + cs]).ravel()
    assert np.max(np.abs(full - ref)) / np.max(np.abs(ref)) < 1e-13
    with pytest.raises(ValueError):
        gplan.separable_weights(np.random.default_rng(0).uniform(1, 2, (4, 5)))


def test_gauss_kernel_and_filter_matrices_host(golden):
    """Host side of the degree-wise filters: Gauss kernel table and the diagonal filter matrices
    (no GPU involved)."""
    import grates_b200 as gb
    from grates_b200 import kernel as gk
    g = golden("degreewise_filters")
    for radius in (0.0, 150.0, 500.0):
        np.testing.assert_array_equal(gk.Gauss(radius).coefficients(0, 200).ravel(), g["gauss_w_%d" % radius])
    np.testing.assert_array_equal(gk.Gauss(300.0).coefficients(1020, 1030).ravel()[0:5], g["gauss_w_300_ext"][0:5])
    with pytest.raises(ValueError):
        gk.Gauss(-1.0)
    np.testing.assert_array_equal(np.diag(gb.Gaussian(300.0).matrix(2, 9)), g["gauss_matrix_300_2_9"])
    m = gb.Butterworth(5, 12).matrix(1, 12)
    np.testing.assert_array_equal(np.diag(m), g["butter_matrix_5_12"])
    assert np.count_nonzero(m - np.diag(np.diag(m))) == 0
    w = gb.Gaussian(500.0).degree_weights(40)
    assert w[0] == 1.0 and w[1] == 1.0 and w[2] == g["gauss_w_500"][2]
    with pytest.raises(TypeError):
        gb.Gaussian(300.0).filter(np.zeros((5, 5)))


def _reference_standin():
    """The classes of the reference package (akvas/grates) that install() rebinds, reduced to what the wrappers read
    and write.  Their own PotentialCoefficients.to_grid is the numpy port of the reference's (oracle/sh_oracle.py,
    pinned to the reference's outputs by test_oracle_golden.py); the other rebound methods only have to exist."""
    import copy
    import types
    from oracle import sh_oracle as orc

    def not_exercised(self, *args, **kwargs):
        raise AssertionError("not exercised by this test")

    class PotentialCoefficients:
        def __init__(self, GM=orc.GM_DEFAULT, R=orc.R_DEFAULT):
            self.GM, self.R, self.anm, self.epoch = GM, R, np.zeros((1, 1)), None

        def copy(self):
            return copy.deepcopy(self)

        def to_grid(self, grid, kernel='ewh'):
            og = orc.OracleGrid(grid.meridians, grid.parallels, a=grid.semimajor_axis, f=grid.flattening)
            out = grid.copy()
            out.values = orc.synthesis(self.anm, og, kernel, self.GM, self.R).ravel()
            return out

    class RegularGrid:
        def __init__(self, meridians, parallels, area=None, a=orc.A_GRS80, f=orc.F_GRS80):
            og = orc.OracleGrid(meridians, parallels, area, a, f)
            self.meridians, self.parallels, self.area = og.meridians, og.parallels, og.areas.ravel()
            self.semimajor_axis, self.flattening, self.values, self.epoch = a, f, None, None

        def copy(self):
            return copy.deepcopy(self)

        to_potential_coefficients = covariance_propagation = not_exercised

    class GeographicGrid(RegularGrid):
        def __init__(self, dlon=0.5, dlat=0.5, a=orc.A_GRS80, f=orc.F_GRS80):
            og = orc.geographic_grid(dlon, dlat, a, f)
            super().__init__(og.meridians, og.parallels, og.areas, a, f)

    class IrregularGrid:
        covariance_propagation = not_exercised

    class Filter:
        filter = not_exercised

    class RadialBasisFunctions:
        to_potential_coefficients = not_exercised

    return types.SimpleNamespace(
        gravityfield=types.SimpleNamespace(PotentialCoefficients=PotentialCoefficients, gridded_rms=not_exercised,
                                           RadialBasisFunctions=RadialBasisFunctions),
        grid=types.SimpleNamespace(RegularGrid=RegularGrid, GeographicGrid=GeographicGrid, IrregularGrid=IrregularGrid),
        filter=types.SimpleNamespace(**{name: type(name, (Filter,), {}) for name in
                                        ("OrderWiseFilter", "Gaussian", "Butterworth", "GeneralMatrix", "VDK")}))


def test_install_rebinds_reference_methods_and_has_no_cpu_fallback(golden):
    """grates_b200.install() rebinds the hot methods of the reference's own classes (SURVEY 8b); without a
    CUDA device the rebound methods raise instead of computing on the CPU; uninstall() restores them.  The reference
    package is not part of this repository, so the classes patched here are a stand-in (_reference_standin) with the
    attributes the wrappers use, not the reference's own: this test does not show that the wrappers agree with the real
    classes (their copy(), the shape of their area array, ...).  What it pins to the reference is the numbers: the
    stand-in's own to_grid and the rebound one are both compared with the reference's output stored in
    tests/golden/synthesis.npz (make_golden.py, same coefficients, grid and kernel)."""
    import torch
    grates = _reference_standin()
    g = golden("synthesis")
    reference = g["s_ewh"][0].ravel()
    original = grates.gravityfield.PotentialCoefficients.to_grid
    pc = grates.gravityfield.PotentialCoefficients()
    pc.anm = g["s_anm"][0].copy()
    grid = grates.grid.GeographicGrid(dlon=10.0, dlat=10.0)
    expected = pc.to_grid(grid, "ewh").values.copy()
    assert maxnorm_err(expected, reference) < 4e-15
    try:
        gb.install(grates)
        assert grates.gravityfield.PotentialCoefficients.to_grid is not original
        assert len(gb.installed()) == 11
        if not torch.cuda.is_available():
            with pytest.raises(Exception) as err:
                pc.to_grid(grid, "ewh")
            assert "CUDA" in str(err.value) or "cuda" in str(err.value)
        else:
            out = pc.to_grid(grid, "ewh")
            assert type(out) is type(grid) and out is not grid and grid.values is None
            assert maxnorm_err(out.values, reference) < 1e-12
    finally:
        gb.uninstall()
    assert grates.gravityfield.PotentialCoefficients.to_grid is original and not gb.installed()
    np.testing.assert_array_equal(pc.to_grid(grid, "ewh").values, expected)


def test_general_matrix_host_logic(golden):
    """GeneralMatrix: constructor checks and the degree-range remapping of matrix() (filter.py:445-509), VDK matrix."""
    import grates_b200 as gb
    g = golden("dense_filters")
    flt = gb.GeneralMatrix(g["W_2_10"], 2, 10)
    np.testing.assert_array_equal(flt.matrix(2, 10), g["W_2_10"])
    np.testing.assert_array_equal(flt.matrix(0, 12), g["matrix_0_12"])
    np.testing.assert_array_equal(flt.matrix(4, 8), g["matrix_4_8"])
    with pytest.raises(ValueError):
        gb.GeneralMatrix(np.zeros((3, 4)), 0, 1)
    with pytest.raises(ValueError):
        gb.GeneralMatrix(np.zeros((5, 5)), 0, 1)
    vdk = gb.VDK(g["normals_2_10"], 2, 10, 1e2, 2.0)
    np.testing.assert_allclose(vdk.matrix(2, 10), g["vdk_matrix"], rtol=1e-12, atol=1e-15)


def test_blocked_normals_vdk_blocks_match_reference(golden):
    """BlockedNormalsVDK (reference filter.py:352-427): block extraction and regularised solves are host work;
    the assembled filter matrix equals the reference's bit for bit."""
    import grates_b200 as gb
    g = golden("dense_filters")
    flt = gb.filter.BlockedNormalsVDK(g["normals_2_10"], 2, 10, 1e2, 2.0)
    np.testing.assert_array_equal(flt.matrix(0, 10), g["blocked_vdk_matrix"])
