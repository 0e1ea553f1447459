"""GPU parity tests: the CUDA path (through the Python host mirror -> ctypes -> C ABI) against
(a) golden outputs of the unmodified reference (tests/golden) and (b) the CPU oracle on the same
seeded inputs.  Parity metric: max|d| / max|ref| (BASELINE.md section 3); tolerance 1e-12
(1e-10 at degree >= 180) as stated by BASELINE.json north_star; Legendre tables bit-exact."""
import datetime

import numpy as np
import pytest

from conftest import maxnorm_err

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

KERNELS = ("ewh", "obp", "potential", "geoid", "surface_density", "anomaly", "deformation", "uplift")
TOL = 1e-12


@pytest.fixture(scope="module")
def gb():
    import grates_b200
    grates_b200._lib.require_device()
    return grates_b200


@pytest.fixture(scope="module")
def orc():
    from oracle import sh_oracle
    return sh_oracle


def _pc(gb, anm, GM=None, R=None):
    pc = gb.PotentialCoefficients() if GM is None else gb.PotentialCoefficients(GM, R)
    pc.anm = np.array(anm, dtype=float)
    return pc


# ------------------------------------------------------------------------------ Legendre
def test_legendre_bit_exact_vs_reference(gb, golden):
    g = golden("l1_numerics")
    for N in (5, 40):
        out = gb.utilities.legendre_functions(N, g["colat"])
        np.testing.assert_array_equal(out, g["legendre_%d" % N])
    out = gb.utilities.legendre_functions(200, g["colat"][::4])
    np.testing.assert_array_equal(out, g["legendre_200"])       # includes polar underflow to denormals / 0


def test_legendre_scaled_table(gb, orc):
    grid = gb.GeographicGrid(5.0, 5.0)
    plan = gb.get_plan(grid, 30, "ewh")
    colat, kn = orc.kn_table("ewh", 30, grid.parallels)
    ref = orc._scale_packed_by_degree(orc.legendre_functions(30, colat), kn)
    np.testing.assert_array_equal(plan.legendre_table(scaled=True).cpu().numpy(), ref)
    np.testing.assert_array_equal(plan.kn, kn)


# ------------------------------------------------------------------------------ synthesis
def test_synthesis_config1_golden(gb, golden):
    g = golden("synthesis")
    grid = gb.GeographicGrid(1.0, 1.0)
    out = _pc(gb, g["c1_anm"]).to_grid(grid, "ewh")
    assert type(out) is gb.GeographicGrid and out.value_array.shape == (180, 360)
    assert grid.value_array is None                                # input grid untouched
    assert maxnorm_err(out.value_array, g["c1_ewh"]) < TOL
    assert out.values.shape == (64800,)


@pytest.mark.parametrize("name", KERNELS)
def test_synthesis_kernels_golden(gb, golden, name):
    g = golden("synthesis")
    grid = gb.GeographicGrid(10.0, 10.0)
    batch = gb.to_grid_batch(g["s_anm"], grid, name)
    assert batch.shape == (3, 18, 36)
    assert maxnorm_err(batch, g["s_" + name]) < TOL
    for e in range(3):
        single = _pc(gb, g["s_anm"][e]).to_grid(grid, name).value_array
        assert maxnorm_err(single, g["s_" + name][e]) < TOL


def test_synthesis_variants_golden(gb, golden):
    g = golden("synthesis")
    grid = gb.GeographicGrid(10.0, 10.0)
    out = _pc(gb, g["s_anm"][0], g["s_gmr"][0], g["s_gmr"][1]).to_grid(grid, "ewh")
    assert maxnorm_err(out.value_array, g["s_ewh_gmr"]) < TOL
    from oracle import sh_oracle as orc
    anm20 = orc.synthetic_coefficients(20, 0)
    gg = gb.GaussGrid(24)
    out = _pc(gb, anm20).to_grid(gg, "ewh")
    assert type(out) is gb.GaussGrid and maxnorm_err(out.value_array, g["gauss_ewh"]) < TOL
    rg = gb.RegularGrid(g["reg_meridians"], g["reg_parallels"])
    assert maxnorm_err(_pc(gb, anm20).to_grid(rg, "geoid").value_array, g["reg_geoid"]) < TOL
    assert maxnorm_err(_pc(gb, np.array([[1.0]])).to_grid(grid, "potential").value_array, g["deg0_potential"]) < TOL
    rp = gb.RegularGrid(g["hi_meridians"], g["hi_parallels"])
    hi = _pc(gb, g["hi_anm"]).to_grid(rp, "ewh").value_array       # degree 200, polar underflow
    assert np.all(np.isfinite(hi)) and maxnorm_err(hi, g["hi_ewh"]) < 1e-10


def test_synthesis_default_grid_and_epoch(gb, orc):
    pc = _pc(gb, orc.synthetic_coefficients(8, 3))
    out = pc.to_grid()                                             # default 0.5 degree grid, ewh
    assert out.value_array.shape == (360, 720)
    ref = orc.synthesis(pc.anm, orc.geographic_grid(0.5, 0.5), "ewh")
    assert maxnorm_err(out.value_array, ref) < TOL
    g = gb.GeographicGrid(5.0, 5.0)
    g.epoch = datetime.datetime(2005, 1, 1)
    assert pc.to_grid(g, "ewh").epoch == g.epoch


def test_synthesis_tensor_core_vs_plain_kernel(gb, orc, monkeypatch):
    """The DMMA stage-2 kernel and the one-thread-per-output kernel agree to rounding."""
    grid = gb.GeographicGrid(2.0, 2.0)
    anm = np.stack([orc.synthetic_coefficients(45, e) for e in range(5)])
    fast = gb.to_grid_batch(anm, grid, "ewh")
    monkeypatch.setenv("GB_NAIVE_STAGE2", "1")
    plain = gb.to_grid_batch(anm, grid, "ewh")
    monkeypatch.delenv("GB_NAIVE_STAGE2")
    assert maxnorm_err(fast, plain) < 1e-14
    monkeypatch.setenv("GB_SIMPLE_STAGE1", "1")            # FMA stage 1 instead of the DMMA one
    simple = gb.to_grid_batch(anm, grid, "ewh")
    monkeypatch.delenv("GB_SIMPLE_STAGE1")
    assert maxnorm_err(fast, simple) < 1e-14
    ref = np.stack([orc.synthesis(a, orc.geographic_grid(2.0, 2.0), "ewh") for a in anm])
    assert maxnorm_err(fast, ref) < TOL


@pytest.mark.parametrize("nmax,dlon,E", [(0, 5.0, 1), (1, 5.0, 2), (2, 45.0, 1), (45, 1.5, 5), (96, 0.5, 2), (97, 1.0, 3)])
def test_synthesis_symmetric_vs_general_path(gb, orc, monkeypatch, nmax, dlon, E):
    """Meridian counts divisible by 8 take the four-fold symmetric stage 2; it must agree with the
    general contraction (GB_NO_SYMMETRY=1) to rounding and with the oracle to tolerance."""
    grid = gb.GeographicGrid(dlon, 3.0)
    anm = np.stack([orc.synthetic_coefficients(nmax, e) for e in range(E)])
    anm[:, 0, 0] = 1e-6
    if nmax >= 1:
        anm[:, 1, 0], anm[:, 1, 1], anm[:, 0, 1] = 2e-6, -3e-6, 4e-6
    sym = gb.to_grid_batch(anm, grid, "ewh")
    # 16-byte store path: an output 16- but not 32-byte aligned (two doubles past the start of its allocation)
    plan, x = gb.get_plan(grid, nmax, "ewh"), torch.as_tensor(anm).cuda()
    aligned = plan.synthesis(x)
    narrow = torch.empty(aligned.numel() + 2, dtype=torch.float64, device="cuda")[2:].view(aligned.shape)
    assert narrow.data_ptr() % 32 == 16
    assert plan.synthesis(x, out=narrow) is narrow and torch.equal(narrow, aligned)
    monkeypatch.setenv("GB_NO_SYMMETRY", "1")
    gen = gb.to_grid_batch(anm, grid, "ewh")
    monkeypatch.delenv("GB_NO_SYMMETRY")
    assert maxnorm_err(sym, gen) < 2e-13
    og = orc.geographic_grid(dlon, 3.0)
    ref = np.stack([orc.synthesis(a, og, "ewh") for a in anm])
    assert maxnorm_err(sym, ref) < TOL and maxnorm_err(gen, ref) < TOL


@pytest.mark.parametrize("nmax,dlat,E", [(1, 30.0, 1), (2, 45.0, 3), (15, 10.0, 2), (16, 6.0, 41), (47, 2.0, 90), (96, 0.5, 2), (120, 1.0, 3), (120, 0.25, 2), (60, 0.25, 130)])
def test_synthesis_equator_fold_vs_unfolded(gb, orc, monkeypatch, nmax, dlat, E):
    """Grids that mirror about the equator run the Legendre recursion for the northern parallels only (declared
    shortcut, gb_plan_is_folded).  White spectra, zonal and full, are the worst case for the hemisphere asymmetry of the
    reference's own cos(theta) table: the folded result must stay within tolerance of the oracle and agree with the
    unfolded stage (GB_NO_FOLD=1) to rounding."""
    grid, og = gb.GeographicGrid(4 * dlat if dlat < 20 else dlat, dlat), None
    og = orc.geographic_grid(4 * dlat if dlat < 20 else dlat, dlat)
    plan = gb.get_plan(grid, nmax, "potential")
    assert plan.folded == (nmax >= 1)
    rng = np.random.default_rng(nmax)
    anm = rng.standard_normal((E, nmax + 1, nmax + 1))
    anm[0] = 0.0
    anm[0, :, 0] = rng.standard_normal(nmax + 1)            # zonal only: largest at the poles
    folded = gb.to_grid_batch(anm, grid, "potential")
    monkeypatch.setenv("GB_NO_FOLD", "1")
    plain = gb.to_grid_batch(anm, grid, "potential")
    monkeypatch.delenv("GB_NO_FOLD")
    ref = np.stack([orc.synthesis(a, og, "potential") for a in anm[:2]])
    assert maxnorm_err(plain[:2], ref) < TOL
    assert maxnorm_err(folded[:2], ref) < TOL
    for e in range(E):
        assert maxnorm_err(folded[e], plain[e]) < 5e-13


def test_equator_fold_is_gated_on_measured_asymmetry(gb, orc):
    """On a 0.25 degree grid one parallel next to the pole fails the gate (the reference's colatitudes there differ
    between the hemispheres by more than it allows): its tile of 32 parallels per hemisphere stays with the unfolded
    stage, the rest is folded.  Grids that are not mirror images are not folded at all."""
    lib = gb._lib.load()
    half = gb.get_plan(gb.GeographicGrid(0.5, 0.5), 96, "ewh")
    assert half.folded and lib.gb_plan_is_folded(half._handle) == 1              # no polar cap needed
    quarter = gb.get_plan(gb.GeographicGrid(1.0, 0.25), 60, "ewh")
    assert quarter.folded and lib.gb_plan_is_folded(quarter._handle) == 2         # one 32-parallel cap per pole
    par = gb.GeographicGrid(10.0, 10.0).parallels.copy()
    par[3] += 1e-9
    assert not gb.get_plan(gb.RegularGrid(gb.GeographicGrid(10.0, 10.0).meridians, par), 8, "ewh").folded
    assert not gb.get_plan(gb.RegularGrid(gb.GeographicGrid(10.0, 10.0).meridians, par[:-1]), 8, "ewh").folded   # odd count
    # a parallel in the second tile of 32 that fails the gate: two polar-cap tiles per pole, still exact
    grid, og = _two_cap_grid(gb, orc)
    assert lib.gb_plan_is_folded(gb.get_plan(grid, 60, "ewh")._handle) == 3
    anm = np.stack([orc.synthetic_coefficients(60, e) for e in range(2)])
    ref = np.stack([orc.synthesis(a, og, "ewh") for a in anm])
    assert maxnorm_err(gb.to_grid_batch(anm, grid, "ewh"), ref) < TOL


def _two_cap_grid(gb, orc):
    """0.5 degree parallels (1 degree meridians) with parallel 40 moved by 1e-9: it fails the fold gate, so the first
    two tiles of 32 parallels per hemisphere run unfolded (gb_plan_is_folded == 3).  Returns the grid and its oracle."""
    base = gb.GeographicGrid(1.0, 0.5)
    par = base.parallels.copy()
    par[40] += 1e-9
    return gb.RegularGrid(base.meridians, par), orc.OracleGrid(base.meridians, par)


@pytest.mark.parametrize("E", [11, 55, 70, 100])         # the 64-, 120-, 80- and 240-column tilings
def test_stage1_recursion_matches_table(gb, orc, monkeypatch, E):
    """Without the plan's Legendre table (over its memory budget; GB_S1_ONTHEFLY=1 forces it) the Legendre stage runs the
    recursion inside the kernel and lays its ring stages out like the table: the results are bit-identical on folded
    grids with and without polar caps and on unfolded grids with an even and an odd number of parallels."""
    lib = gb._lib.load()
    geo3 = gb.GeographicGrid(3.0, 3.0)
    # grid, degree, GB_NO_FOLD, gb_plan_is_folded (1: folded, 2 / 3: folded with one / two polar-cap tiles per pole)
    cases = ((geo3, 40, False, 1), (gb.GeographicGrid(1.0, 0.25), 60, False, 2), (_two_cap_grid(gb, orc)[0], 60, False, 3),
             (geo3, 40, True, 1), (gb.RegularGrid(geo3.meridians, geo3.parallels[:-1]), 40, False, 0))
    rng = np.random.default_rng(E)
    for grid, N, no_fold, folded in cases:
        assert lib.gb_plan_is_folded(gb.get_plan(grid, N, "ewh")._handle) == folded
        x = torch.as_tensor(rng.standard_normal((E, N + 1, N + 1))).cuda()
        if no_fold:
            monkeypatch.setenv("GB_NO_FOLD", "1")
        table = gb.to_grid_batch(x, grid, "ewh")
        monkeypatch.setenv("GB_S1_ONTHEFLY", "1")
        rec = gb.to_grid_batch(x, grid, "ewh")
        monkeypatch.delenv("GB_S1_ONTHEFLY")
        monkeypatch.delenv("GB_NO_FOLD", raising=False)
        assert torch.equal(table, rec), (grid.parallels.size, N, no_fold)
    flt = gb.OrderWiseFilter(orc.synthetic_filter_blocks(40))
    x = torch.as_tensor(rng.standard_normal((E, 41, 41))).cuda()
    table = gb.to_grid_batch(x, geo3, "ewh", orderwise_filter=flt)
    monkeypatch.setenv("GB_S1_ONTHEFLY", "1")
    assert torch.equal(gb.to_grid_batch(x, geo3, "ewh", orderwise_filter=flt), table)


@pytest.mark.parametrize("nmax,dlon,dlat,E", [(1, 30.0, 30.0, 1), (2, 90.0, 45.0, 2), (17, 7.5, 4.0, 7),
                                              (33, 3.0, 3.0, 2), (96, 1.0, 0.5, 3)])
def test_synthesis_ragged_shapes_vs_oracle(gb, orc, nmax, dlon, dlat, E):
    grid = gb.GeographicGrid(dlon, dlat)
    anm = np.stack([orc.synthetic_coefficients(nmax, e) for e in range(E)])
    if nmax < 2:
        anm[:, 0, 0] = 1.0
    out = gb.to_grid_batch(anm, grid, "ewh")
    og = orc.geographic_grid(dlon, dlat)
    ref = np.stack([orc.synthesis(a, og, "ewh") for a in anm])
    assert maxnorm_err(out, ref) < TOL


def test_synthesis_odd_meridian_count(gb, orc):
    mer = np.linspace(-3.0, 3.0, 37)
    par = np.linspace(1.4, -1.4, 9)
    anm = orc.synthetic_coefficients(12, 1)
    out = _pc(gb, anm).to_grid(gb.RegularGrid(mer, par), "potential").value_array
    assert maxnorm_err(out, orc.synthesis(anm, orc.OracleGrid(mer, par), "potential")) < TOL


def test_synthesis_headline_shape_properties(gb, orc):
    """BASELINE config 2 at full size (degree 96 -> 0.5 deg, 240 epochs): device-resident batch.
    The oracle checks 3 epochs directly; the rest through linearity and batch-independence."""
    E, N = 240, 96
    grid = gb.GeographicGrid(0.5, 0.5)
    anm = np.stack([orc.synthetic_coefficients(N, e) for e in range(E)])
    dev = torch.device("cuda")
    x = torch.as_tensor(anm).to(dev)
    out = gb.to_grid_batch(x, grid, "ewh")
    assert out.is_cuda and tuple(out.shape) == (E, 360, 720)
    og = orc.geographic_grid(0.5, 0.5)
    for e in (0, 117, 239):
        assert maxnorm_err(out[e].cpu().numpy(), orc.synthesis(anm[e], og, "ewh")) < TOL
    # batch independence: any sub-batch gives bit-identical rows
    sub = gb.to_grid_batch(x[100:103].contiguous(), grid, "ewh")
    assert torch.equal(sub, out[100:103])
    # linearity: synth(a x_p + b x_q) = a synth(x_p) + b synth(x_q)
    mix = (0.3 * x[5] - 1.7 * x[200])[None].contiguous()
    lin = 0.3 * out[5] - 1.7 * out[200]
    assert maxnorm_err(gb.to_grid_batch(mix, grid, "ewh")[0].cpu().numpy(), lin.cpu().numpy()) < 1e-13
    # host-buffer entry point agrees with the device one
    host = gb.to_grid_batch(anm[:40], grid, "ewh")
    assert isinstance(host, np.ndarray) and np.array_equal(host, out[:40].cpu().numpy())


def test_synthesis_shard_sizes_are_bit_identical(gb, orc):
    """The strong-scaling shards of config 2 (240 / G epochs per GPU) run other tilings than the full batch: 64-column
    items with the CTAs spread over the SMs (30 epochs), one 120-column tile (45 and 60 epochs), 240-column tiles (120),
    and a pack kernel that fetches whole rows with bulk copies.  Every shard must reproduce the rows of the full batch
    bit for bit -- also when the coefficient buffer starts on an odd double, where the bulk copies start one double
    early and the first / last row of the buffer fall back to plain loads."""
    E, N = 240, 96
    grid = gb.GeographicGrid(0.5, 0.5)
    anm = np.stack([orc.synthetic_coefficients(N, e) for e in range(E)])
    x = torch.as_tensor(anm).cuda()
    full = gb.to_grid_batch(x, grid, "ewh")
    for n, e0 in ((30, 0), (30, 210), (45, 17), (60, 180), (120, 120), (1, 239), (33, 5), (41, 100)):
        sub = gb.to_grid_batch(x[e0:e0 + n].contiguous(), grid, "ewh")
        assert torch.equal(sub, full[e0:e0 + n]), (n, e0)
    L = N + 1
    for n in (30, 60):
        flat = torch.zeros(n * L * L + 1, dtype=torch.float64, device="cuda")
        odd = flat[1:].view(n, L, L)
        assert odd.data_ptr() % 16 == 8
        odd.copy_(x[7:7 + n])
        assert torch.equal(gb.to_grid_batch(odd, grid, "ewh"), full[7:7 + n]), n


def test_synthesis_more_than_two_giga_outputs(gb, orc):
    """2 100 epochs on a 0.25 degree grid are 2.18e9 output values (17 GB) and 1.5e6 rows of the spectral intermediate:
    every index that could overflow 32 bits does.  Rows from the start, the middle and the very end of the batch must be
    bit-identical to the same epochs synthesised as a small batch."""
    free, _ = torch.cuda.mem_get_info()
    if free < 40e9:
        pytest.skip("needs 40 GB of free device memory")
    E, N = 2100, 60
    grid = gb.GeographicGrid(0.25, 0.25)
    base = np.stack([orc.synthetic_coefficients(N, e) for e in range(7)])
    x = torch.as_tensor(base).cuda().repeat(E // 7, 1, 1) * torch.linspace(0.5, 1.5, E, dtype=torch.float64, device="cuda")[:, None, None]
    out = gb.to_grid_batch(x, grid, "ewh")
    assert out.numel() > 2**31 and tuple(out.shape) == (E, 720, 1440)
    for e0 in (0, 1047, E - 3):
        sub = gb.to_grid_batch(x[e0:e0 + 3].contiguous(), grid, "ewh")
        assert torch.equal(sub, out[e0:e0 + 3]), e0
    og = orc.geographic_grid(0.25, 0.25)
    assert maxnorm_err(out[E - 1].cpu().numpy(), orc.synthesis(x[E - 1].cpu().numpy(), og, "ewh")) < TOL
    # the analysis of the same 2.18e9 values: the round trip returns the coefficients, the last epochs as a small batch agree
    back = gb.analysis_batch(out, grid, 0, N, "ewh", device_output=True)
    assert float((back - x).abs().max() / x.abs().max()) < 1e-11
    sub = gb.analysis_batch(out[E - 3:].contiguous(), grid, 0, N, "ewh", device_output=True)
    assert maxnorm_err(sub.cpu().numpy(), back[E - 3:].cpu().numpy()) < 1e-14
    del out, back
    gb.clear_plan_cache()               # the 17 GB analysis workspace goes with the plan
    torch.cuda.empty_cache()


def test_time_series_and_rms(gb, orc):
    data = []
    for e in range(6):
        pc = _pc(gb, orc.synthetic_coefficients(20, e))
        pc.epoch = datetime.datetime(2002, 4, 15) + datetime.timedelta(days=30.4375 * (5 - e))
        data.append(pc)
    ts = gb.TimeSeries(data)
    assert ts.epochs() == sorted(ts.epochs())
    grid = gb.GeographicGrid(5.0, 5.0)
    vals = ts.to_grid(grid, "ewh")
    og = orc.geographic_grid(5.0, 5.0)
    ref = np.stack([orc.synthesis(d.anm, og, "ewh") for _, d in ts.items()])
    assert maxnorm_err(vals, ref) < TOL
    np.testing.assert_array_equal(ts.to_array(), orc.ravel_coefficients(np.stack([d.anm for _, d in ts.items()])))
    rms = gb.gridded_rms(ts, ts.epochs(), "ewh", grid)
    assert maxnorm_err(rms.value_array, np.sqrt((ref ** 2).mean(axis=0))) < TOL


# ------------------------------------------------------------------------------ analysis
def test_analysis_golden(gb, golden):
    g = golden("analysis")
    for name in ("ewh", "potential"):
        for lo, hi in ((0, 12), (2, 12), (3, 9)):
            grid = gb.GeographicGrid(10.0, 10.0)
            grid.values = g["in_" + name].ravel().copy()
            pc = grid.to_potential_coefficients(lo, hi, name)
            assert isinstance(pc, gb.PotentialCoefficients) and pc.anm.shape == (hi + 1, hi + 1)
            assert maxnorm_err(pc.anm, g["anm_%s_%d_%d" % (name, lo, hi)]) < TOL
    gg = gb.GaussGrid(14)
    gg.values = g["gauss_in"].ravel().copy()
    assert maxnorm_err(gg.to_potential_coefficients(0, 10, "ewh").anm, g["gauss_anm_0_10"]) < TOL
    rg = gb.RegularGrid(g["reg_meridians"], g["reg_parallels"])
    rg.values = g["reg_in"].ravel().copy()
    assert maxnorm_err(rg.to_potential_coefficients(0, 8, "geoid").anm, g["reg_anm_0_8"]) < 1e-11


def test_analysis_round_trip_batch(gb, orc):
    N, E = 60, 5
    grid = gb.GeographicGrid(1.0, 1.0)
    anm = np.stack([orc.synthetic_coefficients(N, e) for e in range(E)])
    vals = gb.to_grid_batch(anm, grid, "ewh")
    back = gb.analysis_batch(vals, grid, 0, N, "ewh")
    assert back.shape == (E, N + 1, N + 1)
    assert maxnorm_err(back, anm) < 1e-11
    ref = orc.analysis_separable(vals[:2], orc.geographic_grid(1.0, 1.0), 0, N, "ewh")
    assert maxnorm_err(back[:2], ref) < TOL
    dev = gb.analysis_batch(torch.as_tensor(vals).cuda(), grid, 2, N, "ewh", device_output=True)
    assert dev.is_cuda and float(dev[:, :2, :2].abs().max()) == 0.0


@pytest.mark.parametrize("nmax,dlon,dlat", [(30, 1.5, 3.0), (12, 10.0, 10.0), (50, 2.0, 1.0)])
def test_analysis_paths_agree(gb, orc, monkeypatch, nmax, dlon, dlat):
    """Tensor-core longitude stage (four-fold folded where the meridians allow, plain otherwise)
    against the FMA cross-check kernel and the oracle."""
    grid = gb.GeographicGrid(dlon, dlat)
    og = orc.geographic_grid(dlon, dlat)
    rng = np.random.default_rng(5)
    vals = rng.standard_normal((3,) + og.shape)
    ref = orc.analysis_separable(vals, og, 1, nmax, "potential")
    results = {}
    # "hostops": the latitude operators solved with numpy on the host instead of the device Cholesky path
    for tag, env in (("default", {}), ("nosym", {"GB_NO_SYMMETRY": "1"}), ("simple", {"GB_SIMPLE_ANALYSIS": "1"}),
                     ("hostops", {"GB_ANALYSIS_HOST_OPERATORS": "1"})):
        gb.clear_plan_cache()
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        results[tag] = gb.analysis_batch(vals, grid, 1, nmax, "potential")
        for k in env:
            monkeypatch.delenv(k)
    gb.clear_plan_cache()
    for tag, out in results.items():
        assert maxnorm_err(out, ref) < TOL, tag
    assert maxnorm_err(results["default"], results["hostops"]) < 1e-13


def test_dense_operators_golden(gb, golden):
    g = golden("analysis")
    grid = gb.GeographicGrid(30.0, 30.0)
    A = grid.synthesis_matrix(1, 4, "ewh")
    assert A.shape == (72, 24) and maxnorm_err(A, g["synthesis_matrix_1_4"]) < TOL
    F = grid.analysis_matrix(0, 4, "ewh")
    assert F.shape == (25, 72) and maxnorm_err(F, g["analysis_matrix_0_4"]) < TOL
    A0 = grid.synthesis_matrix(0, 4, "ewh")
    np.testing.assert_allclose(F @ A0, np.eye(25), atol=1e-10)          # analysis o synthesis = identity
    c2, s2 = grid.synthesis_matrix_per_order(2, 1, 4, "ewh", 3.9860044150e+14, 6.3781363000e+06)
    np.testing.assert_array_equal(c2, A[:, [4 + 3 - 1, 9 + 3 - 1, 16 + 3 - 1]])
    np.testing.assert_array_equal(s2, A[:, [4 + 4 - 1, 9 + 4 - 1, 16 + 4 - 1]])
    z = grid.synthesis_matrix_per_order(0, 1, 4, "ewh", 3.9860044150e+14, 6.3781363000e+06)
    np.testing.assert_array_equal(z, A[:, [0, 3, 8, 15]])


def test_analysis_errors(gb):
    grid = gb.GeographicGrid(10.0, 10.0)
    with pytest.raises(ValueError):
        grid.to_potential_coefficients(0, 8)                      # no values
    grid.values = np.zeros(grid.point_count)
    with pytest.raises(ValueError):
        grid.to_potential_coefficients(0, 18)                     # N >= nlon / 2
    rng = np.random.default_rng(0)
    bad = gb.RegularGrid(grid.meridians, grid.parallels, rng.uniform(1, 2, (18, 36)))
    bad.values = np.zeros(bad.point_count)
    with pytest.raises(ValueError):
        bad.to_potential_coefficients(0, 8)                       # non-separable area weights


# ------------------------------------------------------------------------------ covariance
def test_covariance_golden(gb, golden):
    g = golden("covariance")
    grid = gb.GeographicGrid(15.0, 15.0)
    std = grid.covariance_propagation(g["sigma"], 0, 8, "ewh")
    assert std.shape == (288,) and maxnorm_err(std, g["std_ewh_0_8"]) < TOL
    np.testing.assert_array_equal(grid.values, std)               # reference also stores the std-devs
    std = gb.GeographicGrid(15.0, 15.0).covariance_propagation(g["sigma"][4:, 4:], 2, 8, "potential")
    assert maxnorm_err(std, g["std_potential_2_8"]) < TOL
    std = gb.GaussGrid(10).covariance_propagation(g["sigma"], 0, 8, "geoid")
    assert maxnorm_err(std, g["std_gauss_geoid"]) < TOL


def test_covariance_vs_oracle_and_row_blocks(gb, orc):
    N = 30
    sigma = orc.synthetic_covariance(N, rank=24)
    grid = gb.GeographicGrid(4.0, 6.0)
    og = orc.geographic_grid(4.0, 6.0)
    ref = orc.covariance_propagation(sigma, og, 0, N, "ewh")
    std = grid.covariance_propagation(sigma, 0, N, "ewh")
    assert maxnorm_err(std, ref) < TOL
    plan = gb.get_plan(grid, N, "ewh")
    s = torch.as_tensor(sigma).cuda()
    parts = [plan.covariance_propagation(s, 0, r0, 10) for r0 in (0, 10, 20)]   # row-block sharding
    assert maxnorm_err(torch.cat(parts).cpu().numpy().ravel(), ref) < TOL
    var = plan.covariance_propagation(s, 0, take_sqrt=False).cpu().numpy().ravel()
    assert maxnorm_err(var, ref ** 2) < TOL
    # closed form: Sigma = I  ->  var_p = sum_a F_pa^2
    eye = torch.eye((N + 1) ** 2, dtype=torch.float64, device="cuda")
    v = plan.covariance_propagation(eye, 0, take_sqrt=False).cpu().numpy()
    P = orc.ravel_coefficients(orc._scale_packed_by_degree(orc.legendre_functions(N, plan.colat), plan.kn))
    T = orc.ravel_coefficients(orc.trigonometric_functions(N, grid.meridians))
    assert maxnorm_err(v, (P ** 2) @ (T ** 2).T) < TOL
    with pytest.raises(ValueError):
        plan.covariance_propagation(s[:-1, :-1], 0)
    # both code paths (order-block pairs k <= k' only / full matrix) agree on a symmetric matrix
    full = plan.covariance_propagation(s, 0, symmetric=False).cpu().numpy().ravel()
    half = plan.covariance_propagation(s, 0, symmetric=True).cpu().numpy().ravel()
    assert maxnorm_err(full, ref) < TOL and maxnorm_err(half, ref) < TOL


def test_covariance_equator_fold_and_mirrored_blocks(gb, orc, monkeypatch):
    """The first contraction runs for the northern parallels only (parity classes of n - m, S +- D): folded against
    unfolded against the oracle, GB_COV_MIRRORED row blocks bit-identical to the full grid, odd parallel counts, a
    min_degree that shifts the parity of the first row of the low orders."""
    for (N, dlon, dlat, nmin) in ((24, 5.0, 5.0, 0), (30, 6.0, 4.0, 3), (17, 9.0, 9.0, 2)):
        grid, og = gb.GeographicGrid(dlon, dlat), orc.geographic_grid(dlon, dlat)
        sigma = orc.synthetic_covariance(N, rank=20)[nmin * nmin:, nmin * nmin:]
        ref = orc.covariance_propagation(sigma, og, nmin, N, "ewh") ** 2
        plan = gb.get_plan(grid, N, "ewh")
        s = torch.as_tensor(np.ascontiguousarray(sigma)).cuda()
        for sym in (True, False):
            monkeypatch.delenv("GB_COV_NO_FOLD", raising=False)
            folded = plan.covariance_propagation(s, nmin, take_sqrt=False, symmetric=sym).cpu().numpy()
            monkeypatch.setenv("GB_COV_NO_FOLD", "1")
            unfolded = plan.covariance_propagation(s, nmin, take_sqrt=False, symmetric=sym).cpu().numpy()
            monkeypatch.delenv("GB_COV_NO_FOLD", raising=False)
            assert maxnorm_err(folded.ravel(), ref) < TOL and maxnorm_err(unfolded.ravel(), ref) < TOL
            nl, a, b = plan.nlat, 1, max(2, plan.nlat // 2 - 1)
            both = plan.covariance_propagation(s, nmin, a, b - a, take_sqrt=False, symmetric=sym, mirrored=True).cpu().numpy()
            np.testing.assert_array_equal(both[:b - a], folded[a:b])
            np.testing.assert_array_equal(both[b - a:], folded[nl - b:nl - a])
        with pytest.raises(ValueError):
            plan.covariance_propagation(s, nmin, plan.nlat // 2, 2, mirrored=True)     # reaches across the equator
    for nl in (10, 11):                  # Gauss grids; 11: the equator is its own mirror image
        sigma = orc.synthetic_covariance(8, rank=8)
        std = gb.GaussGrid(nl).covariance_propagation(sigma, 0, 8, "geoid")
        assert maxnorm_err(std, orc.covariance_propagation(sigma, orc.gauss_grid(nl), 0, 8, "geoid")) < TOL


def test_octant_stage2_matches_quadrant_and_oracle(gb, orc, monkeypatch):
    """Eight-fold longitude symmetry (meridian count divisible by 16): the octant kernel against the four-fold kernel
    (GB_S2_QUADRANT=1), the direct contraction (GB_NO_SYMMETRY=1) and the oracle; whole and half tiles, ragged last
    column tile (90 and 18 octant meridians), grids whose meridian count keeps the four-fold kernel."""
    for (N, dlon, dlat, E, octant) in ((96, 0.5, 1.5, 5, True), (40, 2.5, 2.0, 40, True), (20, 7.5, 5.0, 2, True),
                                       (31, 2.5, 6.0, 130, True), (60, 1.0, 3.0, 4, False)):
        grid, og = gb.GeographicGrid(dlon, dlat), orc.geographic_grid(dlon, dlat)
        plan = gb.get_plan(grid, N, "ewh")
        assert plan.octant == octant and plan.symmetric
        anm = np.stack([orc.synthetic_coefficients(N, e) for e in range(min(E, 3))] * ((E + 2) // 3))[:E]
        x = torch.as_tensor(anm).cuda()
        v8 = plan.synthesis(x)
        monkeypatch.setenv("GB_S2_QUADRANT", "1")
        v4 = plan.synthesis(x)
        monkeypatch.delenv("GB_S2_QUADRANT")
        monkeypatch.setenv("GB_NO_SYMMETRY", "1")
        v1 = plan.synthesis(x)
        monkeypatch.delenv("GB_NO_SYMMETRY")
        ref = np.stack([orc.synthesis(a, og, "ewh") for a in anm[:3]]).reshape(-1, plan.nlat, plan.nlon)
        for v in (v8, v4, v1):
            assert maxnorm_err(v[:ref.shape[0]].cpu().numpy(), ref) < TOL
        assert maxnorm_err(v8.cpu().numpy(), v4.cpu().numpy()) < 1e-13
        if E > 3:
            assert torch.equal(v8[3], v8[0])          # repeated epochs: every row tile gives the same bits


def test_ravel_batch_matches_reference_ordering(gb, orc, golden):
    """Device ravel (utilities.py:310-360) against the reference's TimeSeries.to_array ordering."""
    g = golden("filters")
    out = gb.ravel_batch(g["ts_anm_sorted"]).cpu().numpy()
    np.testing.assert_array_equal(out, g["ts_array"])
    x = np.stack([orc.synthetic_coefficients(31, e) for e in range(3)])
    for nmin in (0, 2, 31):
        np.testing.assert_array_equal(gb.ravel_batch(torch.as_tensor(x).cuda(), nmin).cpu().numpy(),
                                      orc.ravel_coefficients(x, nmin, 31))
    with pytest.raises(ValueError):
        gb.ravel_batch(x, 40)


def test_basin_variances(gb, orc):
    """Variance of area-weighted basin means, w' A S A' w: adjoint synthesis through the analysis kernels,
    device ravel, batched quadratic forms; against the dense oracle."""
    N = 12
    sigma = orc.synthetic_covariance(N, rank=12)
    grid, og = gb.GeographicGrid(10.0, 10.0), orc.geographic_grid(10.0, 10.0)
    rng = np.random.default_rng(21)
    masks = rng.uniform(size=(11, grid.point_count)) < 0.25        # more than eight: two passes over Sigma
    masks[0, :] = True
    for nmin in (0, 2):
        s = sigma[nmin * nmin:, nmin * nmin:]
        ref = orc.basin_variances(s, og, masks, nmin, N, "ewh")
        var = gb.basin_variances(s, grid, masks, nmin, N, "ewh", take_sqrt=False)
        assert maxnorm_err(var, ref) < TOL
        std = gb.basin_variances(torch.as_tensor(s).cuda(), grid, masks.reshape(11, 18, 36), nmin, N, "ewh")
        assert maxnorm_err(std, np.sqrt(ref)) < TOL
    # the functional of the global mean is the degree-0 term only (up to the ellipsoidal factors)
    vec = gb.utilities.ravel_coefficients(np.arange(169.0).reshape(13, 13))
    with pytest.raises(ValueError):
        gb.basin_variances(sigma, grid, np.zeros((1, grid.point_count), dtype=bool), 0, N, "ewh")
    with pytest.raises(ValueError):
        gb.basin_variances(sigma[:-1, :-1], grid, masks, 0, N, "ewh")
    assert vec.shape == (169,)


def test_filtered_covariance_propagation(gb, orc):
    """diag(A F S F' A') with the filter applied to the Legendre factor must equal the reference's way:
    F = filter.matrix(nmin, nmax) (filter.py:72-92, :193-222), S_f = F S F', then grid.py:792-839."""
    N = 18
    sigma = orc.synthetic_covariance(N, rank=16)
    grid = gb.GeographicGrid(6.0, 6.0)
    og = orc.geographic_grid(6.0, 6.0)
    blocks = orc.synthetic_filter_blocks(24)                    # filter reaches beyond the field's degree
    flt = gb.OrderWiseFilter(blocks)
    for nmin in (0, 2):
        F = orc.orderwise_filter_matrix(blocks, nmin, N)
        np.testing.assert_array_equal(F, flt.matrix(nmin, N))
        s = sigma[nmin * nmin:, nmin * nmin:]
        ref = orc.covariance_propagation(F @ s @ F.T, og, nmin, N, "ewh")
        std = gb.GeographicGrid(6.0, 6.0).covariance_propagation(s, nmin, N, "ewh", spatial_filter=flt)
        assert maxnorm_err(std, ref) < TOL
    for iso in (gb.Gaussian(400.0), gb.Butterworth(3, 10)):
        D = iso.matrix(0, N)
        ref = orc.covariance_propagation(D @ sigma @ D.T, og, 0, N, "ewh")
        std = grid.covariance_propagation(sigma, 0, N, "ewh", spatial_filter=iso)
        assert maxnorm_err(std, ref) < TOL
    with pytest.raises(ValueError):
        grid.covariance_propagation(sigma, 0, N, "ewh", spatial_filter=gb.OrderWiseFilter(orc.synthetic_filter_blocks(10)))
    with pytest.raises(TypeError):
        grid.covariance_propagation(sigma, 0, N, "ewh", spatial_filter=object())


def test_covariance_nonsymmetric_matrix_uses_full_path(gb, orc):
    """diag(F S F') only sees the symmetric part of S; a visibly non-symmetric S must be detected and
    propagated with the full matrix (the reference multiplies whatever it is given, grid.py:833-835)."""
    from grates_b200 import plan as gplan
    N = 20
    sigma = orc.synthetic_covariance(N, rank=16)
    rng = np.random.default_rng(7)
    skew = np.triu(rng.standard_normal(sigma.shape), 1) * np.abs(sigma).max() * 0.3
    ns = sigma + skew - skew.T                             # antisymmetric perturbation: variances unchanged
    s = torch.as_tensor(ns).cuda()
    assert not gplan._looks_symmetric(s) and gplan._looks_symmetric(torch.as_tensor(sigma).cuda())
    grid = gb.GeographicGrid(6.0, 6.0)
    plan = gb.get_plan(grid, N, "ewh")
    var = plan.covariance_propagation(s, 0, take_sqrt=False).cpu().numpy().ravel()
    og = orc.geographic_grid(6.0, 6.0)
    ref = orc.covariance_propagation(sigma, og, 0, N, "ewh") ** 2
    assert maxnorm_err(var, ref) < 1e-10                   # cancellation of the antisymmetric part (30 % of max|S|)
    wrong = plan.covariance_propagation(s, 0, take_sqrt=False, symmetric=True).cpu().numpy().ravel()
    assert maxnorm_err(wrong, ref) > 1e-3                  # the half path really relies on symmetry


# ------------------------------------------------------------------------------ irregular point sets
def test_irregular_synthesis_golden(gb, golden, orc):
    g = golden("synthesis")
    ig = gb.IrregularGrid(g["irr_lon"], g["irr_lat"])
    out = _pc(gb, g["irr_anm"]).to_grid(ig, "ewh")
    assert type(out) is gb.IrregularGrid and out.values.shape == (700,) and ig.values is None
    assert maxnorm_err(out.values, g["irr_ewh"]) < TOL
    # batched, other kernel, against the oracle
    rng = np.random.default_rng(3)
    lon, lat = rng.uniform(-np.pi, np.pi, 1111), rng.uniform(-1.57, 1.57, 1111)
    anm = np.stack([orc.synthetic_coefficients(40, e) for e in range(11)])
    vals = gb.to_grid_batch(anm, gb.IrregularGrid(lon, lat), "geoid")
    ref = np.stack([orc.synthesis_points(a, lon, lat, "geoid") for a in anm])
    assert vals.shape == (11, 1111) and maxnorm_err(vals, ref) < TOL


def test_irregular_synthesis_epoch_batch_on_gemm(gb, orc, monkeypatch):
    """Sixteen or more epochs at arbitrary points run as design tiles x DMMA GEMM (gb_points.cu); point count not a
    multiple of the tile, more than one epoch tile; against the oracle and against the per-point kernel."""
    rng = np.random.default_rng(31)
    npts, N, E = 1500, 33, 131
    lon, lat = rng.uniform(-np.pi, np.pi, npts), rng.uniform(-1.57, 1.57, npts)
    anm = np.stack([orc.synthetic_coefficients(N, e) for e in range(E)])
    grid = gb.IrregularGrid(lon, lat)
    vals = gb.to_grid_batch(anm, grid, "ewh")
    assert vals.shape == (E, npts)
    for e in (0, 64, 130):
        assert maxnorm_err(vals[e], orc.synthesis_points(anm[e], lon, lat, "ewh")) < TOL
    monkeypatch.setenv("GB_POINTS_SIMPLE", "1")
    simple = gb.to_grid_batch(anm, grid, "ewh")
    monkeypatch.delenv("GB_POINTS_SIMPLE")
    assert maxnorm_err(vals, simple) < 1e-13


def test_irregular_covariance_golden(gb, golden, orc):
    g = golden("covariance")
    ig = gb.IrregularGrid(g["irr_lon"], g["irr_lat"])
    std = ig.covariance_propagation(g["sigma"], 0, 8, "ewh")
    assert std.shape == (300,) and maxnorm_err(std, g["std_irr_ewh"]) < TOL
    np.testing.assert_array_equal(ig.values, std)
    # larger: odd coefficient count, min_degree > 0, point count not a multiple of the tile
    N, nmin = 24, 2
    sigma = orc.synthetic_covariance(N, rank=16)[nmin * nmin:, nmin * nmin:]
    rng = np.random.default_rng(9)
    lon, lat = rng.uniform(-np.pi, np.pi, 777), rng.uniform(-1.57, 1.57, 777)
    std = gb.IrregularGrid(lon, lat).covariance_propagation(sigma, nmin, N, "potential")
    ref = orc.covariance_propagation_points(sigma, lon, lat, nmin, N, "potential")
    assert maxnorm_err(std, ref) < TOL
    # triangle path (symmetric Sigma) and full path agree; an antisymmetric perturbation needs the full path
    pp = gb.get_points_plan(gb.IrregularGrid(lon, lat), N, "potential")
    sd = torch.as_tensor(sigma).cuda()
    half = pp.covariance_propagation(sd, nmin, symmetric=True).cpu().numpy()
    full = pp.covariance_propagation(sd, nmin, symmetric=False).cpu().numpy()
    assert maxnorm_err(half, ref) < TOL and maxnorm_err(full, ref) < TOL
    skew = np.triu(rng.standard_normal(sigma.shape), 1) * np.abs(sigma).max() * 0.2
    auto = pp.covariance_propagation(torch.as_tensor(sigma + skew - skew.T).cuda(), nmin).cpu().numpy()
    assert maxnorm_err(auto, ref) < 1e-10
    # the direct point kernel and the structured regular-grid kernel agree on a regular grid
    grid = gb.GeographicGrid(12.0, 9.0)
    reg = grid.covariance_propagation(sigma, nmin, N, "potential")
    pts = gb.IrregularGrid(grid.longitude, grid.latitude).covariance_propagation(sigma, nmin, N, "potential")
    assert maxnorm_err(pts, reg) < TOL


# ------------------------------------------------------------------------------ filter
def test_orderwise_filter_golden(gb, golden):
    g = golden("filters")
    blocks = [g["block_%02d" % i] for i in range(25)]
    flt = gb.OrderWiseFilter(blocks)
    for tag in ("12", "9"):
        pc = _pc(gb, g["in_" + tag])
        out = flt.filter(pc)
        assert isinstance(out, gb.PotentialCoefficients) and out is not pc
        assert maxnorm_err(out.anm, g["out_" + tag]) < 1e-14
        np.testing.assert_array_equal(out.anm[0:2, 0:2], g["in_" + tag][0:2, 0:2])
    np.testing.assert_array_equal(flt.matrix(2, 9), g["matrix_2_9"])
    with pytest.raises(ValueError):
        flt.filter(_pc(gb, np.zeros((14, 14))))
    with pytest.raises(TypeError):
        flt.filter(np.zeros((5, 5)))


def test_degreewise_filters_golden_and_fused_synthesis(gb, orc, golden):
    """Gaussian / Butterworth filters (filter.py:31-130): filtered coefficients are bit-identical to the
    reference (one multiplication per coefficient), and weights fused into the synthesis give the same
    grid as filtering first."""
    g = golden("degreewise_filters")
    pc = _pc(gb, g["in_40"])
    for radius in (0.0, 150.0, 500.0):
        np.testing.assert_array_equal(gb.Gaussian(radius).filter(pc).anm, g["gauss_out_%d" % radius])
    for order, cutoff in ((2, 30), (5, 12)):
        np.testing.assert_array_equal(gb.Butterworth(order, cutoff).filter(pc).anm, g["butter_out_%d_%d" % (order, cutoff)])
    np.testing.assert_array_equal(pc.anm, g["in_40"])                      # input untouched
    grid = gb.GeographicGrid(6.0, 6.0)
    flt = gb.Gaussian(300.0)
    vals = flt.filter(pc).to_grid(grid, "ewh").value_array
    assert maxnorm_err(vals, g["ewh_gauss300_in40"]) < TOL
    batch = np.stack([g["in_40"], 2.0 * g["in_40"], g["gauss_out_150"]])
    fused = gb.to_grid_batch(batch, grid, "ewh", degree_weights=flt.degree_weights(40))
    plain = gb.to_grid_batch(flt.filter_batch(batch), grid, "ewh")
    np.testing.assert_array_equal(fused, plain)                            # same products, same kernels
    assert maxnorm_err(fused[0], g["ewh_gauss300_in40"]) < TOL
    dev = flt.filter_batch(torch.as_tensor(batch).cuda())
    assert dev.is_cuda
    np.testing.assert_array_equal(dev.cpu().numpy()[0], orc.degreewise_filter(g["in_40"], orc.gauss_weights(300.0, 40), 2))
    with pytest.raises(ValueError):
        gb.to_grid_batch(batch, grid, "ewh", degree_weights=np.ones(7))


def test_device_reductions_gridded_rms_and_statistics(gb, orc):
    """Consumers that keep the grids on the device: gridded_rms (gravityfield.py:1143-1172) and the
    area-weighted statistics of Grid.mean / rms / std (grid.py:174-260) for a whole batch."""
    import datetime
    N, E = 20, 5
    grid = gb.GeographicGrid(6.0, 6.0)
    og = orc.geographic_grid(6.0, 6.0)
    anm = np.stack([orc.synthetic_coefficients(N, e) for e in range(E)])
    ref = np.stack([orc.synthesis(a, og, "ewh") for a in anm])
    data = []
    for e in range(E):
        pc = _pc(gb, anm[e])
        pc.epoch = datetime.datetime(2002, 4, 15) + datetime.timedelta(days=30.4375 * e)
        data.append(pc)
    ts = gb.TimeSeries(data)
    rms = gb.gridded_rms(ts, ts.epochs(), "ewh", grid)
    assert maxnorm_err(rms.values, np.sqrt(np.sum(ref ** 2, axis=0) / E).ravel()) < TOL
    vals = gb.to_grid_batch(torch.as_tensor(anm).cuda(), grid, "ewh")
    rng = np.random.default_rng(3)
    for mask in (None, rng.uniform(size=grid.point_count) < 0.3):
        st = gb.grid_statistics(vals, grid, mask)
        for e in range(E):
            g1 = grid.copy()
            g1.values = ref[e].ravel()
            assert abs(st["mean"][e] - g1.mean(mask)) < 1e-12 * np.abs(ref[e]).max()
            assert abs(st["rms"][e] - g1.rms(mask)) < 1e-12 * np.abs(ref[e]).max()
            assert abs(st["std"][e] - g1.std(mask)) < 1e-12 * np.abs(ref[e]).max()
    host = gb.grid_statistics(ref, grid)                     # numpy input, same numbers
    np.testing.assert_allclose(host["rms"], st_all_rms(ref, grid), rtol=1e-12)


def st_all_rms(ref, grid):
    w = np.asarray(grid.area).ravel()
    return np.sqrt((ref.reshape(ref.shape[0], -1) ** 2 @ w) / w.sum())


def test_install_wrappers_on_gpu(gb, orc, golden):
    """The wrappers of grates_b200.install() on the GPU.  The reference package cannot travel to the GPU box,
    so a stand-in with the reference's class layout (subclasses of the mirror classes, private block list
    under the reference's mangled name) is patched; the CPU suite patches the real package."""
    import types

    class PC(gb.PotentialCoefficients):
        def copy(self):
            new = PC(self.GM, self.R)
            new.anm = self.anm.copy()
            new.epoch = self.epoch
            return new

    class RG(gb.RegularGrid):
        def copy(self):
            g2 = RG.__new__(type(self))
            RG.__init__(g2, self.meridians.copy(), self.parallels.copy(), self._areas.copy(), self._a, self._f)
            g2.epoch = self.epoch
            return g2

    class GG(RG):
        def __init__(self, dlon=0.5, dlat=0.5):
            base = gb.GeographicGrid(dlon, dlat)
            RG.__init__(self, base.meridians, base.parallels, base._areas, base._a, base._f)

    class IG(gb.IrregularGrid):
        pass

    class OWF:
        def __init__(self, blocks):
            self._OrderWiseFilter__array = blocks

        def filter(self, gravityfield):
            raise AssertionError("not rebound")

    class GA(OWF):
        def __init__(self, radius):
            self.radius = radius

    class BW(OWF):
        def __init__(self, order, cutoff_degree):
            self.order, self.cutoff_degree = order, cutoff_degree

    class RBF:
        def __init__(self, point_distribution, K, min_degree, max_degree):
            self._RadialBasisFunctions__K = K
            self._RadialBasisFunctions__min_degree, self._RadialBasisFunctions__max_degree = min_degree, max_degree
            self.point_distribution, self.GM, self.R, self.epoch = point_distribution, PC().GM, PC().R, None
            self.values = None

        def to_potential_coefficients(self, blocking_factor=256):
            raise AssertionError("not rebound")

    ref = types.SimpleNamespace(
        gravityfield=types.SimpleNamespace(PotentialCoefficients=PC, gridded_rms=None, RadialBasisFunctions=RBF),
        grid=types.SimpleNamespace(RegularGrid=RG, IrregularGrid=IG, GeographicGrid=GG),
        filter=types.SimpleNamespace(OrderWiseFilter=OWF, Gaussian=GA, Butterworth=BW))
    g = golden("degreewise_filters")
    try:
        gb.install(ref)
        pc = PC()
        pc.anm = g["in_40"].copy()
        grid = GG(6.0, 6.0)
        out = pc.to_grid(grid, "ewh")
        assert type(out) is GG and out is not grid
        og = orc.geographic_grid(6.0, 6.0)
        assert maxnorm_err(out.value_array, orc.synthesis(g["in_40"], og, "ewh")) < TOL
        back = out.to_potential_coefficients(2, 20, "ewh")          # 60 meridians resolve up to degree 29
        assert type(back) is PC
        assert maxnorm_err(back.anm, orc.analysis_separable(out.value_array[None], og, 2, 20, "ewh")[0]) < TOL
        filt = GA(500.0).filter(pc)
        assert type(filt) is PC
        np.testing.assert_array_equal(filt.anm, g["gauss_out_500"])
        np.testing.assert_array_equal(BW(2, 30).filter(pc).anm, g["butter_out_2_30"])
        with pytest.raises(TypeError):
            GA(500.0).filter(np.zeros((3, 3)))
        sigma = orc.synthetic_covariance(8, rank=8)
        cg = GG(15.0, 15.0)
        std = cg.covariance_propagation(sigma, 0, 8, "ewh")
        assert maxnorm_err(std, orc.covariance_propagation(sigma, orc.geographic_grid(15.0, 15.0), 0, 8, "ewh")) < TOL
        np.testing.assert_array_equal(cg.values, std)
        rb = golden("radial_basis")
        rbf = RBF(IG(rb["lon"], rb["lat"]), rb["K"], 2, 20)
        rbf.values = rb["values"]
        conv = rbf.to_potential_coefficients()
        assert type(conv) is PC and maxnorm_err(conv.anm, rb["anm"]) < TOL
    finally:
        gb.uninstall()
    assert not gb.installed()


def test_irregular_operators_golden(gb, orc, golden):
    """IrregularGrid.synthesis_matrix(_per_order) from the point-set design kernel, the least-squares analysis operator and
    to_potential_coefficients (reference grid.py:412-443, 477-507, 957-1017) against the reference's outputs."""
    g = golden("irregular_operators")
    grid = gb.IrregularGrid(g["lon"], g["lat"], g["area"])
    A = grid.synthesis_matrix(2, 6, "ewh")
    assert A.shape == (240, 45) and maxnorm_err(A, g["A_2_N_ewh"]) < TOL
    c3, s3 = grid.synthesis_matrix_per_order(3, 2, 6, "ewh", 3.9860044150e+14, 6.3781363000e+06)
    assert maxnorm_err(c3, g["A_m3_cos"]) < TOL and maxnorm_err(s3, g["A_m3_sin"]) < TOL
    F = grid.analysis_matrix(0, 6, "potential")
    assert F.shape == (49, 240) and maxnorm_err(F, g["F_0_N_potential"]) < 1e-10
    grid.values = g["values"]
    back = grid.to_potential_coefficients(2, 6, "ewh")
    assert maxnorm_err(back.anm, g["anm_2_N_ewh"]) < 1e-10
    with pytest.raises(ValueError):
        gb.IrregularGrid(g["lon"], g["lat"]).to_potential_coefficients(0, 4)
    # the dense operator is the point synthesis: A x == to_grid at the points, for a larger, ragged case
    rng = np.random.default_rng(3)
    P, N = 1500, 33
    big = gb.IrregularGrid(rng.uniform(-np.pi, np.pi, P), np.arcsin(rng.uniform(-1, 1, P)))
    anm = orc.synthetic_coefficients(N, 2)
    A = big.synthesis_matrix(0, N, "ewh")
    pc = gb.PotentialCoefficients()
    pc.anm = anm
    np.testing.assert_allclose(A @ orc.ravel_coefficients(anm), pc.to_grid(big, "ewh").values, rtol=0, atol=1e-13 * np.abs(A).max())
    assert maxnorm_err(A[::97], orc.synthesis_matrix_points(big.longitude[::97], big.latitude[::97], 0, N, "ewh")) < TOL


def test_space_kernels_golden_and_batch(gb, orc, golden):
    """AnisotropicKernel.evaluate / evaluate_grid and FilterKernel (kernel.py:576-658, filter.py:575-598): design rows of
    the source points, the dense operator on the filter GEMM, synthesis on the unit sphere."""
    from grates_b200.kernel import AnisotropicKernel
    from grates_b200.filter import FilterKernel
    g = golden("space_kernels")
    ker = AnisotropicKernel(g["K"], 2, 12)
    for i, (slon, slat) in enumerate(g["sources"]):
        pts = ker.evaluate(slon, slat, g["eval_lon"], g["eval_lat"])
        assert pts.shape == (50,) and maxnorm_err(pts, g["points_%d" % i]) < TOL
        grid = ker.evaluate_grid(slon, slat, g["grid_lon"], g["grid_lat"])
        assert grid.shape == (13, 24) and maxnorm_err(grid, g["grid_%d" % i]) < TOL
    both = ker.evaluate_grid_batch(g["sources"][:, 0], g["sources"][:, 1], g["grid_lon"], g["grid_lat"]).cpu().numpy()
    assert maxnorm_err(both, np.stack([g["grid_0"], g["grid_1"]])) < TOL
    fk = FilterKernel(gb.Gaussian(400.0), 2, 12, "ewh")
    assert maxnorm_err(fk.evaluate(0.3, 0.7, g["eval_lon"], g["eval_lat"]), g["gauss_points"]) < TOL
    fo = FilterKernel(gb.OrderWiseFilter([g["block_%d" % i] for i in range(25)]), 2, 12, "potential")
    assert maxnorm_err(fo.evaluate(-2.0, -0.4, g["eval_lon"], g["eval_lat"]), g["orderwise_points"]) < TOL
    np.testing.assert_allclose(fo.modulation_transfer(g["mtf_psi"], 0.2, 0.3, 0.4), g["mtf"], rtol=0, atol=1e-10)
    # footprints of 40 source points on a grid in one call, against the oracle (where the reference's FilterKernel
    # cannot evaluate grids at all)
    rng = np.random.default_rng(12)
    slon, slat = rng.uniform(-np.pi, np.pi, 40), np.arcsin(rng.uniform(-1, 1, 40))
    many = fo.evaluate_grid_batch(slon, slat, g["grid_lon"], g["grid_lat"]).cpu().numpy()
    K3 = orc.filter_kernel_matrix(orc.orderwise_filter_matrix([g["block_%d" % i] for i in range(25)], 2, 12), 2, 12)
    for e in (0, 17, 39):
        assert maxnorm_err(many[e], orc.anisotropic_kernel_evaluate_grid(K3, 2, 12, slon[e], slat[e], g["grid_lon"], g["grid_lat"])) < TOL


def test_covariance_from_normals_feeds_propagation_on_device(gb, orc):
    """Normal-equation matrix -> Sigma = N^-1 on the device -> grid standard deviations, no host round trip of Sigma
    (the dense case of NormalEquations.compute_covariance, lstsq.py:1026-1043, in front of grid.py:792-839)."""
    N = 12
    k = (N + 1) ** 2
    rng = np.random.default_rng(21)
    J = rng.standard_normal((3 * k, k))
    normals = J.T @ J + 1e-3 * np.eye(k)
    sigma = gb.covariance_from_normals(normals)
    assert sigma.is_cuda and tuple(sigma.shape) == (k, k)
    ref_sigma = np.linalg.inv(normals)
    assert maxnorm_err(sigma.cpu().numpy(), ref_sigma) < 1e-10
    grid = gb.GeographicGrid(10.0, 10.0)
    std = grid.covariance_propagation(sigma, 0, N, "ewh")                      # CUDA tensor accepted as is
    assert maxnorm_err(std, orc.covariance_propagation(ref_sigma, orc.geographic_grid(10.0, 10.0), 0, N, "ewh").ravel()) < 1e-9
    pts = gb.IrregularGrid(rng.uniform(-np.pi, np.pi, 300), np.arcsin(rng.uniform(-1, 1, 300)))
    std_p = pts.covariance_propagation(sigma, 0, N, "ewh")
    assert maxnorm_err(std_p, orc.covariance_propagation_points(ref_sigma, pts.longitude, pts.latitude, 0, N, "ewh")) < 1e-9


def test_radial_basis_functions_golden_and_batch(gb, orc, golden):
    """RadialBasisFunctions (gravityfield.py:645-781): the sum over nodal points as a GEMM against the on-the-fly design
    matrix.  Golden vectors of the reference; a batch of value sets over several point blocks against the oracle."""
    g = golden("radial_basis")
    pts = gb.IrregularGrid(g["lon"], g["lat"])
    rbf = gb.RadialBasisFunctions(pts, g["K"], 2, 20)
    rbf.values = g["values"]
    pc = rbf.to_potential_coefficients()
    assert pc.anm.shape == (21, 21) and maxnorm_err(pc.anm, g["anm"]) < TOL
    out = rbf.to_grid(gb.GeographicGrid(6.0, 6.0), "ewh")
    assert maxnorm_err(out.value_array, g["grid_ewh"]) < TOL
    twin = rbf.copy()
    np.testing.assert_array_equal(twin.values, rbf.values)
    M = rbf.to_potential_coefficients_matrix()
    assert M.shape == (21 ** 2 - 4, 700) and maxnorm_err(M[:, ::50], g["matrix_cols"]) < TOL
    np.testing.assert_allclose(orc.unravel_coefficients(M @ g["values"], 2, 20), g["anm"], rtol=0, atol=1e-13 * np.abs(g["anm"]).max())
    # anisotropic basis functions (gravityfield.py:573-642): point adjoint -> dense operator -> synthesis
    abf = gb.AnisotropicBasisFunctions(gb.IrregularGrid(g["lon"][:300], g["lat"][:300]), g["aniso_K"], 2, 10)
    abf.values = g["aniso_values"]
    aout = abf.to_grid(gb.GeographicGrid(10.0, 10.0), "ewh")
    assert maxnorm_err(aout.value_array, g["aniso_grid_ewh"]) < TOL
    rng = np.random.default_rng(8)
    N, P, E = 45, 5000, 130                     # 17 coefficient tiles, two epoch tiles, one block of points (16 384 max)
    lon = rng.uniform(-np.pi, np.pi, P)
    lat = np.arcsin(rng.uniform(-1, 1, P))
    K = rng.uniform(0.5, 1.5, (N + 1, N + 1))
    big = gb.RadialBasisFunctions(gb.IrregularGrid(lon, lat), K, 0, N)
    v = rng.standard_normal((E, P))
    anm = big.to_potential_coefficients_batch(v).cpu().numpy()
    assert anm.shape == (E, N + 1, N + 1)
    for e in (0, 119, 129):
        assert maxnorm_err(anm[e], orc.radial_basis_to_coefficients(K, v[e], lon, lat, N)) < TOL
    for sub in (7, 30):                         # narrower epoch tiles of the GEMM (24 and 48 columns)
        part = big.to_potential_coefficients_batch(v[:sub]).cpu().numpy()
        assert maxnorm_err(part, anm[:sub]) < 1e-14
    # the adjoint identity <A x, v> = <x, A' v> ties it to the point synthesis
    plan = big._points_plan()
    x = torch.as_tensor(rng.standard_normal((3, N + 1, N + 1))).cuda()
    vv = torch.as_tensor(v[:3]).cuda()
    lhs = (plan.synthesis(x) * vv).sum(dim=1)
    rhs = (x * plan.adjoint(vv)).sum(dim=(1, 2))
    np.testing.assert_allclose(lhs.cpu().numpy(), rhs.cpu().numpy(), rtol=1e-11)


def test_dense_matrix_filter_golden_and_batch(gb, orc, golden):
    """GeneralMatrix (filter.py:430-510) as one GEMM over the epoch batch: golden outputs for inputs of equal, lower
    and higher degree than the filter; a larger random case against the oracle."""
    g = golden("dense_filters")
    flt = gb.GeneralMatrix(g["W_2_10"], 2, 10)
    for N in (10, 7, 14):
        pc = _pc(gb, g["in_%d" % N])
        out = flt.filter(pc).anm
        assert out.shape == g["out_%d" % N].shape
        assert maxnorm_err(out, g["out_%d" % N]) < TOL
        np.testing.assert_array_equal(pc.anm, g["in_%d" % N])
    rng = np.random.default_rng(5)
    nmin, nmax, E = 0, 30, 130                                    # K = 961: eight row tiles, two epoch tiles
    k = (nmax + 1) ** 2 - nmin ** 2
    W = 0.5 * np.eye(k) + rng.standard_normal((k, k)) / k
    big = gb.GeneralMatrix(W, nmin, nmax)
    x = np.stack([orc.synthetic_coefficients(nmax, e) for e in range(E)])
    y = big.filter_batch(torch.as_tensor(x).cuda()).cpu().numpy()
    ref = np.stack([orc.dense_filter(W, nmin, nmax, a) for a in x[[0, 64, 129]]])
    assert maxnorm_err(y[[0, 64, 129]], ref) < TOL
    bvdk = gb.filter.BlockedNormalsVDK(g["normals_2_10"], 2, 10, 1e2, 2.0)          # filter.py:352-427
    assert maxnorm_err(bvdk.filter(_pc(gb, g["in_10"])).anm, g["blocked_vdk_out_10"]) < TOL
    vdk = gb.VDK(g["normals_2_10"], 2, 10, 1e2, 2.0)
    out = vdk.filter(_pc(gb, g["in_10"])).anm
    assert maxnorm_err(out, orc.dense_filter(g["vdk_matrix"], 2, 10, g["in_10"])) < 1e-11


def test_orderwise_filter_batch_then_synthesis(gb, orc):
    """BASELINE config 5 in small: block filter over an epoch batch feeding the synthesis."""
    nf, N, E = 40, 36, 11
    blocks = orc.synthetic_filter_blocks(nf)
    flt = gb.OrderWiseFilter(blocks)
    anm = np.stack([orc.synthetic_coefficients(N, e) for e in range(E)])
    out = flt.filter_batch(anm)
    ref = np.stack([orc.orderwise_filter(blocks, a) for a in anm])
    assert maxnorm_err(out, ref) < 1e-14
    dev = flt.filter_batch(torch.as_tensor(anm).cuda())
    assert dev.is_cuda and np.array_equal(dev.cpu().numpy(), out)
    grid = gb.GeographicGrid(3.0, 3.0)
    vals = gb.to_grid_batch(dev, grid, "ewh").cpu().numpy()
    og = orc.geographic_grid(3.0, 3.0)
    assert maxnorm_err(vals, np.stack([orc.synthesis(a, og, "ewh") for a in ref])) < TOL
    # fused: the filter writes into the synthesis workspace (the tiled layout the Legendre stage reads, whether it is fed
    # from the table or runs the recursion); bit-identical to the two calls, on folded and unfolded grids, batches above
    # and below the narrow-tile limit, a filter of higher degree than the data
    x = torch.as_tensor(anm).cuda()
    for g2 in (grid, gb.GeographicGrid(7.0, 5.0), gb.GaussGrid(19)):
        for xe in (x, x[:3], torch.cat([x] * 5), torch.cat([x] * 9)):      # 64-, 120- (55 epochs) and 240-column items
            two = gb.to_grid_batch(flt.filter_batch(xe), g2, "ewh")
            one = gb.to_grid_batch(xe, g2, "ewh", orderwise_filter=flt)
            assert torch.equal(one, two)
    import os
    os.environ["GB_S1_ONTHEFLY"] = "1"
    try:
        assert torch.equal(gb.to_grid_batch(x, grid, "ewh", orderwise_filter=flt), gb.to_grid_batch(dev, grid, "ewh"))
    finally:
        del os.environ["GB_S1_ONTHEFLY"]
    with pytest.raises(ValueError):
        gb.to_grid_batch(x, grid, "ewh", orderwise_filter=gb.OrderWiseFilter(orc.synthetic_filter_blocks(20)))


# ------------------------------------------------------------------------------ API behaviour
def test_api_errors(gb):
    with pytest.raises(ValueError):
        gb.PotentialCoefficients(max_degree=3).to_grid(gb.GeographicGrid(30.0, 30.0), "no_such_kernel")

    with pytest.raises(TypeError):
        gb.PotentialCoefficients(max_degree=3).to_grid(object(), "ewh")
    with pytest.raises(NotImplementedError):
        gb.get_plan(gb.IrregularGrid(np.zeros(3), np.zeros(3)), 3, "ewh")
    plan = gb.get_plan(gb.GeographicGrid(30.0, 30.0), 3, "ewh")
    with pytest.raises(ValueError):
        plan.synthesis(torch.zeros((1, 5, 5), dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        plan.synthesis(torch.zeros((1, 4, 4), dtype=torch.float32, device="cuda"))
    assert plan.synthesis(torch.zeros((0, 4, 4), dtype=torch.float64, device="cuda")).shape == (0, 6, 12)
    assert gb.get_plan(gb.GeographicGrid(30.0, 30.0), 3, "ewh") is plan       # cached


def test_out_buffers_are_checked(gb):
    """A caller-supplied result buffer reaches the kernels as a raw pointer: wrong device, dtype, shape, strides or an
    address that is not 16-byte aligned must raise before anything is launched."""
    grid = gb.GeographicGrid(30.0, 30.0)
    plan = gb.get_plan(grid, 3, "ewh")
    x = torch.zeros((2, 4, 4), dtype=torch.float64, device="cuda")
    good = torch.empty((2, 6, 12), dtype=torch.float64, device="cuda")
    assert plan.synthesis(x, out=good) is good
    for bad in (torch.empty((2, 6, 12), dtype=torch.float64),                      # host tensor
                torch.empty((2, 6, 12), dtype=torch.float32, device="cuda"),
                torch.empty((2, 6, 13), dtype=torch.float64, device="cuda"),
                torch.empty((2, 12, 6), dtype=torch.float64, device="cuda").transpose(1, 2),
                torch.empty(2 * 6 * 12 + 1, dtype=torch.float64, device="cuda")[1:].view(2, 6, 12)):   # 8-byte aligned
        with pytest.raises(ValueError):
            plan.synthesis(x, out=bad)
    # the library itself refuses the misaligned buffer too
    import ctypes
    odd = torch.empty(2 * 6 * 12 + 1, dtype=torch.float64, device="cuda")[1:]
    rc = gb._lib.load().gb_synthesis(plan._handle, ctypes.c_void_p(x.data_ptr()), 2, ctypes.c_void_p(odd.data_ptr()), None)
    assert rc == gb._lib.GB_ERR_ARGUMENT
    plan.set_analysis(0, grid.area.reshape(plan.nlat, plan.nlon))
    with pytest.raises(ValueError):
        plan.analysis(good, out=torch.empty((2, 4, 5), dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        plan.analysis_host(np.zeros((2, 6, 12)), out=np.zeros((2, 4, 4), dtype=np.float32))
    sigma = torch.eye(16, dtype=torch.float64, device="cuda")
    with pytest.raises(ValueError):
        plan.covariance_propagation(sigma, 0, out=torch.empty((6, 11), dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        plan.covariance_propagation(sigma, 0, row0=4, nrows=5)
    with pytest.raises(ValueError):
        gb.Gaussian(300.0).filter_batch(x, out=torch.empty((2, 4, 4), dtype=torch.float64))
    pts = gb.get_points_plan(gb.IrregularGrid(np.linspace(-1, 1, 5), np.linspace(-0.5, 0.5, 5)), 3, "ewh")
    with pytest.raises(ValueError):
        pts.synthesis(x, out=torch.empty((2, 6), dtype=torch.float64, device="cuda"))


def test_calls_on_different_streams_share_one_plan(gb, orc):
    """One plan = one workspace: a call on another stream is ordered behind the previous call's kernels
    (gb_plan_acquire), so back-to-back asynchronous calls from two streams give the serial results."""
    N, E = 40, 48
    grid = gb.GeographicGrid(2.0, 2.0)
    plan = gb.get_plan(grid, N, "ewh")
    xa = torch.as_tensor(np.stack([orc.synthetic_coefficients(N, e) for e in range(E)])).cuda()
    xb = torch.as_tensor(np.stack([orc.synthetic_coefficients(N, 100 + e) for e in range(E)])).cuda()
    want_a, want_b = plan.synthesis(xa).clone(), plan.synthesis(xb).clone()
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    got = []
    for rep in range(6):
        with torch.cuda.stream(s1):
            a = plan.synthesis(xa)
        with torch.cuda.stream(s2):
            b = plan.synthesis(xb)
        got.append((a, b))
    torch.cuda.synchronize()
    for a, b in got:
        assert torch.equal(a, want_a) and torch.equal(b, want_b)


def test_grid_statistics_ignore_values_outside_the_mask(gb):
    """Grid.mean / rms / std select the masked points (grid.py:174-260): a NaN outside the mask must not reach the result."""
    grid = gb.GeographicGrid(10.0, 10.0)
    rng = np.random.default_rng(3)
    vals = rng.standard_normal((3, grid.point_count))
    mask = rng.uniform(size=grid.point_count) < 0.4
    dirty = vals.copy()
    dirty[:, ~mask] = np.nan
    clean, got = gb.grid_statistics(vals, grid, mask), gb.grid_statistics(dirty, grid, mask)
    for key in ("mean", "rms", "std"):
        assert np.all(np.isfinite(got[key])) and np.array_equal(got[key], clean[key])
    g = grid.copy()
    g.values = vals[1]
    assert abs(got["mean"][1] - g.mean(mask)) < 1e-14 and abs(got["rms"][1] - g.rms(mask)) < 1e-14


# ------------------------------------------------------------------------------ covariance producers (SURVEY 8 f4)
def _upper_blocks(index):
    n = int(index[-1])
    mask = np.zeros((n, n), dtype=bool)
    for i in range(len(index) - 1):
        mask[index[i]:index[i + 1], index[i]:] = True
    return mask


def test_block_matrix_golden(gb, golden):
    """Device BlockMatrix against the reference's own block algorithms on a block-sparse SPD matrix with ragged blocks
    (golden vectors of BlockMatrix.cholesky / solve_triangular / multiply_* / sparse_inverse / inverse and
    NormalEquations.compute_covariance, lstsq.py:698-882, 1026-1042)."""
    import copy
    g = golden("normal_equations")
    N, index, rhs = g["N"], g["index"], g["rhs"]
    mask = _upper_blocks(index)
    bm = gb.BlockMatrix.from_array(N, index, index)
    for i in range(6):
        for j in range(i, 6):
            assert bm.is_nonzero(i, j) == bool(g["keep"][i, j])
    assert np.array_equal(bm.to_array(), N)
    assert maxnorm_err(bm.multiply_symmetric(rhs), g["multiply_symmetric"]) < 1e-14
    chol = copy.deepcopy(bm)
    chol.cholesky()
    W = chol.to_array()
    assert maxnorm_err(np.triu(W), g["cholesky"]) < 1e-14 and np.array_equal(np.tril(W[:37, :37], -1), np.zeros((37, 37)))
    assert chol.is_nonzero(1, 3)                                       # fill-in below the extra block, as in the reference
    assert maxnorm_err(chol.solve_triangular(rhs, transpose=True), g["solve_t"]) < 1e-13
    assert maxnorm_err(chol.solve_triangular(rhs, transpose=False), g["solve_n"]) < 1e-13
    assert maxnorm_err(chol.multiply_triangular(rhs), g["multiply_triangular"]) < 1e-14
    sp = copy.deepcopy(chol)
    sp.sparse_inverse()
    assert maxnorm_err(sp.to_array()[mask], g["sparse_inverse"][mask]) < 1e-13
    full = copy.deepcopy(chol)
    full.inverse()
    assert maxnorm_err(full.to_array()[mask], g["inverse"][mask]) < 1e-13
    ne = gb.NormalEquations(copy.deepcopy(bm), rhs[:, 0:1].copy(), 7.5, 4000)
    x = ne.solve()
    assert maxnorm_err(x, np.linalg.solve(N, rhs[:, 0:1])) < 1e-13
    ne = gb.NormalEquations(copy.deepcopy(bm), rhs[:, 0:1].copy(), 7.5, 4000)
    ne.compute_covariance(sparse=False)
    assert ne.status == 'covariance_matrix'
    assert maxnorm_err(ne.matrix.to_array()[mask], g["covariance_dense"][mask]) < 1e-13
    bad = gb.BlockMatrix.from_array(-np.eye(10), np.array([0, 4, 10]), np.array([0, 4, 10]))
    with pytest.raises(np.linalg.LinAlgError):
        bad.cholesky()
    with pytest.raises(ValueError):
        gb.BlockMatrix.from_array(N, index[:-1], index)
    with pytest.raises(ValueError):
        bm[0, 1] = np.zeros((3, 3))


def test_dense_kernels_ragged_shapes(gb):
    """gb_dgemm / gb_dpotrf_upper / gb_dtrsm_upper on shapes that are not multiples of the 64-tile, all transpose
    combinations, strided views (leading dimension > width)."""
    from grates_b200.lstsq import _Ops
    ops = _Ops(None)
    rng = np.random.default_rng(8)
    for (m, n, k) in ((1, 1, 1), (65, 130, 17), (200, 63, 129), (7, 300, 64)):
        for ta in (False, True):
            for tb in (False, True):
                a = rng.standard_normal((k, m) if ta else (m, k))
                b = rng.standard_normal((n, k) if tb else (k, n))
                c = rng.standard_normal((m, n + 5))
                ad, bd, cd = (torch.as_tensor(z).cuda() for z in (a, b, c))
                ops.gemm(ad, bd, cd[:, 2:2 + n], alpha=-0.5, beta=2.0, trans_a=ta, trans_b=tb)
                want = c.copy()
                want[:, 2:2 + n] = -0.5 * (a.T if ta else a) @ (b.T if tb else b) + 2.0 * c[:, 2:2 + n]
                assert maxnorm_err(cd.cpu().numpy(), want) < 1e-14
    for n in (1, 64, 65, 200, 333):
        a = rng.standard_normal((n + 20, n))
        spd = a.T @ a + n * np.eye(n)
        w = ops.cholesky_upper(torch.as_tensor(spd).cuda()).cpu().numpy()
        assert maxnorm_err(w, np.linalg.cholesky(spd).T) < 1e-13
        b = rng.standard_normal((n, 37))
        wd = torch.as_tensor(w).cuda()
        for trans in (False, True):
            x = ops.solve_triangular(wd, torch.as_tensor(b).cuda(), trans=trans).cpu().numpy()
            assert maxnorm_err((w.T if trans else w) @ x, b) < 1e-12
        assert maxnorm_err(ops.inv_gram(wd).cpu().numpy(), np.linalg.inv(spd)) < 1e-12


def test_normals_to_variances_on_the_device(gb, orc):
    """End of the f4 row: normal equations (block matrix on the device) -> compute_covariance -> dense tensor ->
    covariance_propagation, nothing leaves the GPU in between; against the oracle's numpy path."""
    N = 24
    K = (N + 1) ** 2
    rng = np.random.default_rng(6)
    A = rng.standard_normal((3 * K, K)) * (1.0 / (1.0 + np.arange(K)) ** 0.25)[None, :]
    normals = A.T @ A + 1e-3 * np.eye(K)
    ri, ci = gb.BlockMatrix.compute_block_index(normals.shape, 200)
    ne = gb.NormalEquations(gb.BlockMatrix.from_array(normals, ri, ci), rng.standard_normal((K, 1)), 1.0, 3 * K)
    ne.compute_covariance(sparse=False)
    sigma = ne.matrix.symmetrize().to_tensor()
    assert sigma.is_cuda
    want = orc.normal_matrix_inverse(normals)
    assert maxnorm_err(sigma.cpu().numpy(), want) < 1e-10
    grid, og = gb.GeographicGrid(5.0, 5.0), orc.geographic_grid(5.0, 5.0)
    std = gb.get_plan(grid, N, "ewh").covariance_propagation(sigma, 0).cpu().numpy()
    assert maxnorm_err(std, orc.covariance_propagation(want, og, 0, N, "ewh").reshape(std.shape)) < 1e-9


def test_surface_mascons(gb, orc):
    """SurfaceMasCons (gravityfield.py:484-570): container arithmetic and analysis through the grid kernels."""
    grid = gb.GeographicGrid(6.0, 6.0)
    anm = orc.synthetic_coefficients(12, 4)
    field = gb.PotentialCoefficients()
    field.anm = anm
    grid.values = field.to_grid(grid, "ewh").values
    mc = gb.SurfaceMasCons(grid, "ewh")
    back = mc.to_potential_coefficients(0, 12)
    assert maxnorm_err(back.anm, anm) < 1e-12
    twice = (mc + mc) / 2 - mc * 0.5
    assert maxnorm_err(twice.values, 0.5 * mc.values) < 1e-15
    with pytest.raises(TypeError):
        mc + 1.0


# ------------------------------------------------------------------------------ BASELINE full sizes
def test_config3_full_size_round_trip(gb, orc):
    """BASELINE config 3 geometry (degree 180 -> 0.25 deg, 720 x 1440): synthesis against the oracle
    for one epoch (tolerance 1e-10 at degree >= 180), analysis through the round trip (size-independent
    property) and against the separable oracle on one epoch."""
    N, E = 180, 6
    grid, og = gb.GeographicGrid(0.25, 0.25), orc.geographic_grid(0.25, 0.25)
    anm = np.stack([orc.synthetic_coefficients(N, e) for e in range(E)])
    x = torch.as_tensor(anm).cuda()
    vals = gb.to_grid_batch(x, grid, "ewh")
    ref0 = orc.synthesis(anm[0], og, "ewh")
    assert maxnorm_err(vals[0].cpu().numpy(), ref0) < 1e-10
    back = gb.analysis_batch(vals, grid, 0, N, "ewh", device_output=True)
    assert float((back - x).abs().max() / x.abs().max()) < 1e-10
    assert maxnorm_err(back[0].cpu().numpy(), orc.analysis_separable(ref0, og, 0, N, "ewh")) < 1e-10


def test_config4_full_size_properties(gb, orc):
    """BASELINE config 4 at full size (K = 9409 coefficients, 360 x 720 grid): closed form for
    Sigma = I, scaling (std is homogeneous of degree 1/2 in Sigma), row-block sharding and three
    parallels against the oracle."""
    N = 96
    grid, og = gb.GeographicGrid(0.5, 0.5), orc.geographic_grid(0.5, 0.5)
    plan = gb.get_plan(grid, N, "ewh")
    K = (N + 1) ** 2
    eye = torch.eye(K, dtype=torch.float64, device="cuda")
    var = plan.covariance_propagation(eye, 0, take_sqrt=False).cpu().numpy()
    P = orc.ravel_coefficients(orc._scale_packed_by_degree(orc.legendre_functions(N, plan.colat), plan.kn))
    T = orc.ravel_coefficients(orc.trigonometric_functions(N, grid.meridians))
    assert maxnorm_err(var, (P ** 2) @ (T ** 2).T) < TOL
    del eye
    sig_h = orc.synthetic_covariance(N)
    sigma = torch.as_tensor(sig_h).cuda()
    std = plan.covariance_propagation(sigma, 0)
    ref = orc.covariance_propagation(sig_h, og, 0, N, "ewh", rows=[7, 180, 352])
    assert maxnorm_err(std[[7, 180, 352]].cpu().numpy(), ref) < TOL
    std4 = plan.covariance_propagation(sigma * 4.0, 0)
    assert maxnorm_err(std4.cpu().numpy(), 2.0 * std.cpu().numpy()) < 1e-13
    blocks = torch.cat([plan.covariance_propagation(sigma, 0, r0, 45) for r0 in range(0, 360, 45)])   # 8-GPU partition
    assert maxnorm_err(blocks.cpu().numpy(), std.cpu().numpy()) < 1e-13


def test_covariance_propagation_is_bit_reproducible(gb, orc):
    """Every partial sum of the propagation has one writer and the partials are added in a fixed order (no floating-point
    atomics): two runs give bit-identical standard deviations, for the regular-grid path (symmetric and general matrix,
    whole grid and a row block) and for the point-set kernel."""
    N = 60
    grid = gb.GeographicGrid(1.0, 1.0)
    plan = gb.get_plan(grid, N, "ewh")
    sig_h = orc.synthetic_covariance(N)
    sigma = torch.as_tensor(sig_h).cuda()
    for kwargs in ({}, {"symmetric": False}, {"row0": 37, "nrows": 45}):
        first = plan.covariance_propagation(sigma, 0, **kwargs).clone()
        for _ in range(3):
            assert torch.equal(plan.covariance_propagation(sigma, 0, **kwargs), first)
    rng = np.random.default_rng(5)
    pts = gb.IrregularGrid(rng.uniform(-np.pi, np.pi, 700), np.arcsin(rng.uniform(-1, 1, 700)))
    pp = gb.get_points_plan(pts, N, "ewh")
    first = pp.covariance_propagation(sigma, 0).clone()
    for _ in range(3):
        assert torch.equal(pp.covariance_propagation(sigma, 0), first)


def test_config5_filter_then_synthesis_full_degree(gb, orc):
    """BASELINE config 5 geometry (degree 120 -> 0.25 deg) on a reduced epoch count: two epochs against
    the oracle, linearity of filter + synthesis for the batch."""
    N, E = 120, 12
    grid, og = gb.GeographicGrid(0.25, 0.25), orc.geographic_grid(0.25, 0.25)
    blocks = orc.synthetic_filter_blocks(N)
    flt = gb.OrderWiseFilter(blocks)
    anm = np.stack([orc.synthetic_coefficients(N, e) for e in range(E)])
    x = torch.as_tensor(anm).cuda()
    vals = gb.to_grid_batch(flt.filter_batch(x), grid, "ewh")
    for e in (0, E - 1):
        ref = orc.synthesis(orc.orderwise_filter(blocks, anm[e]), og, "ewh")
        assert maxnorm_err(vals[e].cpu().numpy(), ref) < TOL
    mix = (2.0 * x[3] - 0.5 * x[9])[None].contiguous()
    lin = 2.0 * vals[3] - 0.5 * vals[9]
    got = gb.to_grid_batch(flt.filter_batch(mix), grid, "ewh")[0]
    assert maxnorm_err(got.cpu().numpy(), lin.cpu().numpy()) < 1e-13


def test_config3_full_epoch_count(gb, orc):
    """BASELINE config 3 at its real size (degree 180 -> 0.25 deg, ALL 120 epochs: the tilings of the full batch, not a
    reduced one): three epochs against the oracle, every other epoch through batch independence (a sub-batch gives
    bit-identical rows) and linearity; analysis of the 120-epoch batch through the round trip, against the separable
    oracle on one epoch and bit-identical to a sub-batch."""
    N, E = 180, 120
    grid, og = gb.GeographicGrid(0.25, 0.25), orc.geographic_grid(0.25, 0.25)
    anm = np.stack([orc.synthetic_coefficients(N, e) for e in range(E)])
    x = torch.as_tensor(anm).cuda()
    vals = gb.to_grid_batch(x, grid, "ewh")
    assert tuple(vals.shape) == (E, 720, 1440)
    refs = {e: orc.synthesis(anm[e], og, "ewh") for e in (0, 61, 119)}
    for e, ref in refs.items():
        assert maxnorm_err(vals[e].cpu().numpy(), ref) < 1e-10
    for lo, hi in ((0, 2), (57, 64), (113, 120)):
        assert torch.equal(gb.to_grid_batch(x[lo:hi].contiguous(), grid, "ewh"), vals[lo:hi])
    mix = (0.3 * x[5] - 1.7 * x[100])[None].contiguous()
    lin = 0.3 * vals[5] - 1.7 * vals[100]
    assert maxnorm_err(gb.to_grid_batch(mix, grid, "ewh")[0].cpu().numpy(), lin.cpu().numpy()) < 1e-13
    back = gb.analysis_batch(vals, grid, 0, N, "ewh", device_output=True)
    assert float((back - x).abs().max() / x.abs().max()) < 1e-10
    assert maxnorm_err(back[61].cpu().numpy(), orc.analysis_separable(refs[61], og, 0, N, "ewh")) < 1e-10
    sub = gb.analysis_batch(vals[57:64].contiguous(), grid, 0, N, "ewh", device_output=True)
    assert maxnorm_err(sub.cpu().numpy(), back[57:64].cpu().numpy()) < 1e-14


def test_config5_full_epoch_count(gb, orc):
    """BASELINE config 5 at its real size (degree 120 -> 0.25 deg, ALL 500 epochs: 1000 stage-1 columns = four whole
    240-column tiles and a ragged fifth): three epochs of filter + synthesis against the oracle, sub-batches
    bit-identical, linearity."""
    N, E = 120, 500
    grid, og = gb.GeographicGrid(0.25, 0.25), orc.geographic_grid(0.25, 0.25)
    blocks = orc.synthetic_filter_blocks(N)
    flt = gb.OrderWiseFilter(blocks)
    anm = np.stack([orc.synthetic_coefficients(N, e) for e in range(E)])
    x = torch.as_tensor(anm).cuda()
    filt = flt.filter_batch(x)
    vals = gb.to_grid_batch(filt, grid, "ewh")
    assert tuple(vals.shape) == (E, 720, 1440)
    for e in (0, 250, 499):
        want = orc.orderwise_filter(blocks, anm[e])
        assert maxnorm_err(filt[e].cpu().numpy(), want) < 1e-13
        assert maxnorm_err(vals[e].cpu().numpy(), orc.synthesis(want, og, "ewh")) < TOL
    for lo, hi in ((0, 3), (238, 243), (478, 500)):
        sub_f = flt.filter_batch(x[lo:hi].contiguous())
        assert torch.equal(sub_f, filt[lo:hi])
        assert torch.equal(gb.to_grid_batch(sub_f, grid, "ewh"), vals[lo:hi])
    mix = (2.0 * x[3] - 0.5 * x[409])[None].contiguous()
    lin = 2.0 * vals[3] - 0.5 * vals[409]
    got = gb.to_grid_batch(flt.filter_batch(mix), grid, "ewh")[0]
    assert maxnorm_err(got.cpu().numpy(), lin.cpu().numpy()) < 1e-13


def test_degree_360(gb, orc):
    """Degree 360 (tolerance 1e-10 at degree >= 180, north star): synthesis to 0.5 deg against the oracle, block filter,
    analysis round trip on a 0.25 deg grid."""
    N, E = 360, 6
    grid, og = gb.GeographicGrid(0.5, 0.5), orc.geographic_grid(0.5, 0.5)
    anm = np.stack([orc.synthetic_coefficients(N, e) for e in range(E)])
    out = gb.to_grid_batch(torch.as_tensor(anm).cuda(), grid, "ewh")
    assert maxnorm_err(out[3].cpu().numpy(), orc.synthesis(anm[3], og, "ewh")) < 1e-10
    blocks = orc.synthetic_filter_blocks(N)
    f = gb.OrderWiseFilter(blocks).filter_batch(torch.as_tensor(anm[:2]).cuda())
    assert maxnorm_err(f[1].cpu().numpy(), orc.orderwise_filter(blocks, anm[1])) < 1e-13
    grid2 = gb.GeographicGrid(0.25, 0.25)
    v = gb.to_grid_batch(torch.as_tensor(anm[:2]).cuda(), grid2, "ewh")
    back = gb.analysis_batch(v, grid2, 0, N, "ewh", device_output=True)
    assert maxnorm_err(back.cpu().numpy(), anm[:2]) < 1e-10
