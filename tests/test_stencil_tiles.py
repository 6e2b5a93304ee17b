"""Window-kernel stencil tiles: oracle parity of the kernel that derives in-edge indices instead of staging the col table.

When every col word of every 256-neuron tile of a window-kernel lattice equals the one stencil_cols (common.h) gives for the
radius-1 stencil and one lattice-wide release mask, the window kernel stages no col words (Engine::build_win_params,
tile_params_kernel): full warps compute their neighbours' addresses from their own index, border warps compute the col words.
That needs every tile to read its parameter row as well; lattices with per-neuron parameters read the table.  Every case asserts the window path and the count of such tiles (SNN_OPT_STENCIL_TILES): all of
them, or 0 where a tile differs from the stencil (the kernel that reads the table).
"""
import numpy as np
import pytest

import scenarios as SC
import test_param_tiles as TPT
import test_step_paths as TSP
from test_step_paths import kernel_env  # noqa: F401 (fixture)
from test_param_tiles import uniform_lattices  # noqa: F401 (fixture)
from snn_b200 import _capi as K
from snn_b200.dist import LocalStrips
from oracle_api import OracleBackend

pytestmark = pytest.mark.gpu
f32 = np.float32
TILE = 256


def n_tiles(rows, cols):
    return -(-rows * cols // TILE)


def stencil_tiles(lat, win=True):
    """win: the run must have taken the window kernel (False: any other path)."""
    assert (lat._be.get_option(K.OPT_STEP_PATH) == K.STEP_PATH_WIN) == win
    return lat._be.get_option(K.OPT_STENCIL_TILES)


# the bench workload's specialisation (Izhikevich, AMPA, STDP) on ~1 M neurons, so that the deeper ring of the smaller stage
# wraps; without STDP the same lattice is compared bit for bit
@pytest.mark.parametrize("spec", [("izh", "approx_ampa", "stdp"), ("izh", "approx_ampa", None), ("izh", None, None),
                                  ("hh", "destexhe_all", None), ("lif", "expdecay_all", "stdp")], ids=TSP.spec_id)
def test_uniform_lattice_is_all_stencil(spec, uniform_lattices, oracle_lattice_factory):
    built = uniform_lattices()
    rows = 1024 if spec[0] != "hh" else 262
    TSP.run_parity(oracle_lattice_factory, spec, rows, 1000, "grid", TSP.WIN)
    assert stencil_tiles(built[0]) == n_tiles(rows, 1000)


def test_two_release_types(uniform_lattices, oracle_lattice_factory):
    """Every node releases AMPA and NMDA only (release mask 3, not 7): full warps take the per-type path with a uniform mask."""
    def two_types(lat):
        flags = np.zeros((lat.rows * lat.cols, 3), np.uint32)
        flags[:, :2] = 1
        lat.set_field("neurotransmitters$flags", flags)
    built = uniform_lattices(two_types)
    TSP.run_parity(oracle_lattice_factory, ("izh", "approx_all", None), 262, 1000, "grid", TSP.WIN)
    assert stencil_tiles(built[0]) == n_tiles(262, 1000)


@pytest.mark.parametrize("spec", [("lif", None, "stdp"), ("hh", "destexhe_all", None)], ids=TSP.spec_id)
def test_heterogeneous_parameters_read_the_table(spec, kernel_env, oracle_lattice_factory):
    """Per-neuron parameters (no tile reads its parameter row): the kernel that streams every operand, col words included."""
    rows = TSP.win_rows(spec)
    lat = TSP.build(None, spec, rows, 1000, "grid", 5)
    lat.run_lattice(1)
    assert lat._be.get_option(K.OPT_UNIFORM_TILES) == 0
    assert stencil_tiles(lat) == 0


def test_mixed_tiles_read_the_table(uniform_lattices, oracle_lattice_factory):
    """Uniform and non-uniform tiles in one lattice: the two-group kernel, which stages the col words of every tile."""
    built = uniform_lattices(TPT.mixed_edit)
    TSP.run_parity(oracle_lattice_factory, ("izh", None, None), TPT.MIX_ROWS, TPT.MIX_COLS, "grid", TSP.WIN)
    assert 0 < built[0]._be.get_option(K.OPT_UNIFORM_TILES) < n_tiles(TPT.MIX_ROWS, TPT.MIX_COLS)
    assert stencil_tiles(built[0]) == 0


@pytest.mark.parametrize("cols", [37, 100, 255, 257, 1021])
def test_geometry(cols, uniform_lattices, oracle_lattice_factory):
    """Several lattice rows per tile, border warps in the middle of tiles, and a partial last tile."""
    built = uniform_lattices()
    rows = -(-65536 // cols) + 1
    TSP.run_parity(oracle_lattice_factory, ("izh", None, None), rows, cols, "grid", TSP.WIN, seed=cols)
    assert stencil_tiles(built[0]) == n_tiles(rows, cols)


@pytest.mark.parametrize("cols", [1021, 4099])
def test_three_rows(cols, kernel_env, uniform_lattices, oracle_lattice_factory):
    """Every warp touches the top or the bottom row: only border warps."""
    kernel_env(tma=2)
    built = uniform_lattices()
    TSP.run_parity(oracle_lattice_factory, ("izh", "approx_ampa", None), 3, cols, "grid", TSP.WIN, seed=cols)
    assert stencil_tiles(built[0]) == n_tiles(3, cols)


ROWS, COLS = 262, 1000
SPEC = ("izh", "approx_ampa", None)


def pair(oracle_lattice_factory, seed=9):
    a = SC.build_lattice(None, model="izh", rows=ROWS, cols=COLS, seed=seed, chem="approx_ampa", hetero=False)
    b = SC.build_lattice(oracle_lattice_factory, model="izh", rows=ROWS, cols=COLS, seed=seed, chem="approx_ampa", hetero=False)
    b._be.set_option(K.OPT_PARALLEL, 1)
    return a, b


def run_edits(a, b, edits):
    """edits: (edit applied to both lattices or None, window kernel expected, expected stencil tiles), each followed by a run of
    21 or 20 steps (odd and even lengths alternate through the ping-pong parities) compared bit for bit."""
    done = 0
    for k, (edit, win, expect) in enumerate(edits):
        if edit is not None:
            edit(a)
            edit(b)
        steps = 21 if k % 2 == 0 else 20
        a.run_lattice(steps)
        b.run_lattice(steps)
        TSP.compare(a, b, SPEC, done, done + steps)
        done += steps
        assert stencil_tiles(a, win) == expect
    assert b.spike_history.history.sum() > 0


def test_release_types_of_one_node(oracle_lattice_factory, kernel_env):
    """One node stops releasing AMPA: the type bits of its neighbours' col words differ from the stencil's, so a stale check would
    give them AMPA input.  Then the node releases it again."""
    a, b = pair(oracle_lattice_factory)
    n = ROWS * COLS
    node = 100 * COLS + 500
    ones = np.zeros((n, 3), np.uint32)
    ones[:, 0] = 1
    one_off = ones.copy()
    one_off[node] = 0
    tiles = n_tiles(ROWS, COLS)
    run_edits(a, b, [(None, True, tiles),
                     (lambda lat: lat.set_field("neurotransmitters$flags", one_off), True, 0),
                     (lambda lat: lat.set_field("neurotransmitters$flags", ones), True, tiles)])


def test_graph_edits(oracle_lattice_factory, kernel_env):
    """An edge removed (the table is no longer the generator's: the window kernel is not taken), the grid connected again, and
    weights of existing edges edited (the weights stay staged: every tile stays a stencil tile)."""
    a, b = pair(oracle_lattice_factory)
    tiles = n_tiles(ROWS, COLS)
    run_edits(a, b, [(None, True, tiles),
                     (lambda lat: lat.edit_weight((50, 40), (51, 41), None), False, 0),
                     (lambda lat: lat.connect_grid(1, 1.0), True, tiles),
                     (lambda lat: [lat.edit_weight((r, 9), (r + 1, 10), 0.5 + 0.01 * r) for r in range(1, 200, 7)], True, tiles)])


def test_row_strips(kernel_env):
    """Two strips on one device: local neuron 0 is not node 0 and not row 0, and the windows read ghost rows."""
    kernel_env(tma=2)
    rows, cols, world = 2 * 132, 256, 2
    n = rows * cols
    strips = LocalStrips(K.MODEL_IZH, rows, cols, world)
    strips.each(lambda be: be.set_option(K.OPT_HALO_TIMEOUT_MS, 20000))
    ob = OracleBackend(K.MODEL_IZH, 0, 0, rows=rows, cols=cols)
    v = np.random.default_rng(6).uniform(-65, 30, n).astype(f32)
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
        assert be.get_option(K.OPT_STENCIL_TILES) == -(-(own.stop - own.start) // TILE)
    for nm in ("last_firing_time", "is_spiking"):
        assert (strips.get_field(nm) == ob.get_field(0, nm)).all(), nm
    for nm in ("current_voltage", "w_value", "neurotransmitters$t", "receptors$AMPA$r$kinetics$r"):
        np.testing.assert_allclose(strips.get_field(nm), ob.get_field(0, nm), rtol=1e-4, atol=1e-3, err_msg=nm)
    assert (ob.get_field(0, "last_firing_time") >= 0).sum() > n // 4


def test_stencil_tiles_is_read_only():
    lat = SC.build_lattice(None, model="izh", rows=4, cols=4, graph="grid")
    with pytest.raises(K.SnnError) as e:
        lat._be.set_option(K.OPT_STENCIL_TILES, 1)
    assert e.value.status == K.SNN_INVALID_ARGUMENT
    lat.run_lattice(1)
    assert lat._be.get_option(K.OPT_STENCIL_TILES) == 0   # not the window kernel
