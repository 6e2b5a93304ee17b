"""Window-kernel tiles whose neurons share every parameter: oracle parity on the uniform side and at its boundary.

A 256-neuron tile of the window-staged kernel (step_win.cu) whose neurons all have the bit patterns of its first neuron in every
parameter the step reads takes them from one tile row instead of from one stream per parameter (Engine::build_win_params).  The
parity scenarios of test_step_paths randomise parameters per neuron, so every tile there streams; here the lattices are uniform
(Lattice::populate of one neuron, random voltages), and tiles are made non-uniform one by one.  Every case asserts the window
path and how many tiles took the row (SNN_OPT_UNIFORM_TILES), so that a regression to streaming cannot pass silently.
"""
import numpy as np
import pytest

import scenarios as SC
import test_step_paths as TSP
from test_step_paths import kernel_env  # noqa: F401 (fixture)
from snn_b200 import _capi as K
from snn_b200.dist import LocalStrips
from oracle_api import OracleBackend

pytestmark = pytest.mark.gpu
f32 = np.float32
TILE = 256


def n_tiles(rows, cols):
    return -(-rows * cols // TILE)


def uniform_tiles(lat):
    assert lat._be.get_option(K.OPT_STEP_PATH) == K.STEP_PATH_WIN
    return lat._be.get_option(K.OPT_UNIFORM_TILES)


@pytest.fixture
def uniform_lattices(monkeypatch, kernel_env):
    """test_step_paths.build with uniform parameters: scenarios.build_lattice(hetero=False), then edit(lattice) on the device
    lattice and on the oracle alike.  Returns the list of lattices built (the device one first, as run_parity builds them)."""
    built, orig = [], SC.build_lattice

    def install(edit=None):
        def build_lattice(factory, **kw):
            lat = orig(factory, hetero=False, **kw)
            # tonic firing with uniform parameters (the scenarios.build_lattice recipe, one value): Izhikevich b > 0.27 and
            # c_m = 2, leak reversal above threshold.  Without it only the neurons that start near threshold fire, all in the
            # first step, and STDP leaves the weights where they are
            if kw.get("model") == "izh":
                lat.fill_field("b", 0.3)
                lat.fill_field("c_m", 2.0)
            if kw.get("model") == "lif":
                lat.fill_field("e_l", -45.0)
            if edit is not None:
                edit(lat)
            built.append(lat)
            return lat
        monkeypatch.setattr(SC, "build_lattice", build_lattice)
        return built
    return install


UNIFORM_SPECS = [("izh", None, None), ("izh", "approx_ampa", "stdp"), ("hh", "destexhe_all", None), ("lif", "expdecay_all", None),
                 ("bcm_izh", None, "bcm")]


@pytest.mark.parametrize("spec", UNIFORM_SPECS, ids=TSP.spec_id)
def test_uniform_lattice(spec, uniform_lattices, oracle_lattice_factory):
    built = uniform_lattices()
    rows = TSP.win_rows(spec)
    TSP.run_parity(oracle_lattice_factory, spec, rows, 1000, "grid", TSP.WIN)
    assert uniform_tiles(built[0]) == n_tiles(rows, 1000)


@pytest.mark.parametrize("cols", [257, 1021])
def test_uniform_geometry(cols, uniform_lattices, oracle_lattice_factory):
    """Tiles straddle lattice rows, and the last tile is partial: only its valid neurons are compared."""
    built = uniform_lattices()
    rows = -(-65536 // cols) + 1
    TSP.run_parity(oracle_lattice_factory, ("izh", None, "stdp"), rows, cols, "grid", TSP.WIN, seed=cols)
    assert uniform_tiles(built[0]) == n_tiles(rows, cols)


MIX_ROWS, MIX_COLS = 262, 1000
HETERO_TILES = [3, 10, 11, 12, 1023]   # 1023: the last (partial) tile
ONE_D_TILE, ZERO_TILE = 20, 30


def mixed_edit(lat):
    """Whole tiles of random b; one neuron of another tile with a different d (started above threshold, so that it spikes and
    its reset differs); a third tile that differs from its first neuron only in the sign of a zero (a = -0.0 next to +0.0)."""
    n = MIX_ROWS * MIX_COLS
    rng = np.random.default_rng(3)
    b = np.full(n, 0.3, f32)
    for t in HETERO_TILES:
        lo, hi = t * TILE, min(n, (t + 1) * TILE)
        b[lo:hi] = rng.uniform(0.25, 0.36, hi - lo)
    lat.set_field("b", b)
    d = np.full(n, 8.0, f32)
    d[ONE_D_TILE * TILE + 77] = 2.0
    lat.set_field("d", d)
    v = lat.get_field("current_voltage")
    v[ONE_D_TILE * TILE + 77] = 29.0
    lat.set_field("current_voltage", v)
    a = np.zeros(n, f32)
    a[ZERO_TILE * TILE + 5] = -0.0
    lat.set_field("a", a)


def test_mixed_tiles(uniform_lattices, oracle_lattice_factory):
    built = uniform_lattices(mixed_edit)
    TSP.run_parity(oracle_lattice_factory, ("izh", None, None), MIX_ROWS, MIX_COLS, "grid", TSP.WIN)
    a = built[0].get_field("a")
    assert np.signbit(a[ZERO_TILE * TILE + 5]) and not np.signbit(a[ZERO_TILE * TILE + 4])
    assert uniform_tiles(built[0]) == n_tiles(MIX_ROWS, MIX_COLS) - len(HETERO_TILES) - 2


HH_EDITS = {5: "gap_conductance", 9: "receptors$NMDA_mg", 14: "receptors$AMPA$r$kinetics$alpha", 1023: "receptors$GABA_g"}


def hh_mixed_edit(lat):
    """Hodgkin-Huxley with Destexhe kinetics: a tile of random gap conductances, and single neurons whose NMDA Mg, AMPA alpha
    (RCF_MG, RCF_K1: read from the row by uniform tiles, from run-time stage offsets by the others) or GABA g (last, partial
    tile) differ."""
    rng = np.random.default_rng(4)
    for t, name in HH_EDITS.items():
        x = lat.get_field(name)
        if name == "gap_conductance":
            x[t * TILE:(t + 1) * TILE] *= rng.uniform(0.75, 1.25, TILE).astype(f32)
        else:
            x[t * TILE + 3] *= f32(1.5)
        lat.set_field(name, x)


def test_mixed_tiles_hodgkin_huxley(uniform_lattices, oracle_lattice_factory):
    """The mixed-tile kernel with two consumer groups and every receptor parameter kind."""
    built = uniform_lattices(hh_mixed_edit)
    spec = ("hh", "destexhe_all", None)
    rows = TSP.win_rows(spec)
    TSP.run_parity(oracle_lattice_factory, spec, rows, 1000, "grid", TSP.WIN)
    assert uniform_tiles(built[0]) == n_tiles(rows, 1000) - len(HH_EDITS)


def test_edits_between_runs_rebuild_the_tile_rows(oracle_lattice_factory, kernel_env):
    """A parameter of one neuron, then whole model and chemical fields, changed between run calls on the device and in the
    oracle: a stale tile row would step with the old values."""
    spec = ("izh", "approx_ampa", None)
    rows, cols = 262, 1000
    n, tiles = rows * cols, n_tiles(rows, cols)
    a = SC.build_lattice(None, model="izh", rows=rows, cols=cols, seed=9, chem="approx_ampa", hetero=False)
    b = SC.build_lattice(oracle_lattice_factory, model="izh", rows=rows, cols=cols, seed=9, chem="approx_ampa", hetero=False)
    b._be.set_option(K.OPT_PARALLEL, 1)
    d = a.get_field("d")
    d[40 * TILE + 200] = 3.5

    def set_one(lat):
        lat.set_field("d", d)

    def fill_chemical(lat):
        lat.fill_field("receptors$AMPA_g", 2.5)
        lat.fill_field("neurotransmitters$clearance_constant", 0.2)

    def fill_model(lat):
        lat.fill_field("d", 6.0)

    done = 0
    for edit, expect in ((None, tiles), (set_one, tiles - 1), (fill_chemical, tiles - 1), (fill_model, tiles)):
        if edit is not None:
            edit(a)
            edit(b)
        a.run_lattice(20)
        b.run_lattice(20)
        TSP.compare(a, b, spec, done, done + 20)
        done += 20
        assert uniform_tiles(a) == expect
    assert b.spike_history.history.sum() > 0


def test_row_strips_uniform(kernel_env):
    """Two strips on one device (in-process attach), uniform parameters, electrical + AMPA + STDP: boundary tiles import ghost
    rows and still read their tile row."""
    kernel_env(tma=2)   # 33 792 neurons per strip: below the staged kernels' size threshold
    rows, cols, world = 2 * 132, 256, 2
    n = rows * cols
    strips = LocalStrips(K.MODEL_IZH, rows, cols, world)
    strips.each(lambda be: be.set_option(K.OPT_HALO_TIMEOUT_MS, 20000))
    ob = OracleBackend(K.MODEL_IZH, 0, 0, rows=rows, cols=cols)
    v = np.random.default_rng(5).uniform(-65, 30, n).astype(f32)
    flags = np.zeros((n, 3), np.uint32)
    flags[:, 0] = 1
    init = {"current_voltage": v, "b": np.full(n, 0.3, f32), "gap_conductance": np.full(n, 10.0, f32), "c_m": np.full(n, 4.0, f32)}

    def configure(set_field, each):
        for name, arr in init.items():
            set_field(name, arr, 1)
        set_field("neurotransmitters$flags", flags, 3)
        set_field("receptors$flags", flags, 3)

        def opts(be):
            be.connect_grid(0, 1, 0.8)
            be.set_option(K.OPT_ELECTRICAL_SYNAPSE, 1)
            be.set_option(K.OPT_CHEMICAL_SYNAPSE, 1)
            be.set_option(K.OPT_DO_PLASTICITY, 1, 0)
            be.set_plasticity(0, 0.05, 0.04, 4.5, 3.0, 0.1)
        each(opts)

    configure(lambda nm, arr, per: strips.set_field(nm, arr, per), strips.each)
    strips.attach()
    configure(lambda nm, arr, per: ob.set_field(0, nm, np.asarray(arr).reshape(-1)), lambda fn: fn(ob))
    for k in (13, 12):
        strips.run(k)
        ob.run(k)
    for r, be in enumerate(strips.strips):
        assert be.get_option(K.OPT_STEP_PATH) == K.STEP_PATH_WIN
        own = strips.rows_of(r)
        assert be.get_option(K.OPT_UNIFORM_TILES) == -(-(own.stop - own.start) // TILE)
    for nm in ("last_firing_time", "is_spiking"):
        assert (strips.get_field(nm) == ob.get_field(0, nm)).all(), nm
    for nm in ("current_voltage", "w_value", "neurotransmitters$t", "receptors$AMPA$r$kinetics$r"):
        np.testing.assert_allclose(strips.get_field(nm), ob.get_field(0, nm), rtol=1e-4, atol=1e-3, err_msg=nm)
    np.testing.assert_allclose(strips.graph_csr()[2], ob.get_connection_csr()[2], rtol=1e-4, atol=1e-5)
    assert (ob.get_field(0, "last_firing_time") >= 0).sum() > n // 4


def test_uniform_tiles_is_read_only():
    lat = SC.build_lattice(None, model="izh", rows=4, cols=4, graph="grid")
    with pytest.raises(K.SnnError) as e:
        lat._be.set_option(K.OPT_UNIFORM_TILES, 1)
    assert e.value.status == K.SNN_INVALID_ARGUMENT
    lat.run_lattice(1)
    assert lat._be.get_option(K.OPT_UNIFORM_TILES) == 0   # not the window kernel
