"""Graph weight history: Lattice.update_graph_history / LatticeNetwork.update_connecting_graph_history (Graph::update_history,
graph/mod.rs:278-284).  A Lattice records after each step's plasticity (Lattice::iterate, neuron/mod.rs:973-979), a
LatticeNetwork before it (neuron/mod.rs:2565-2576).

CPU tier: the oracle (stepped one timestep at a time by tests/graph_history_oracle.py, which records at the reference's
placements) through the front end.  GPU tier: the device against the oracle, against itself stepped one run(1) at a
time, and with recording on against recording off."""
import numpy as np
import pytest

import scenarios as SC
import snn_b200 as S
from graph_history_oracle import GraphHistoryOracle
from oracle_api import OracleError
from snn_b200 import _capi as K
from test_gpu_parity import build_network

f32 = np.float32
ERRORS = (S.SnnError, OracleError)


@pytest.fixture
def gh_lattice_factory():
    """The CPU oracle in the Lattice role, recording graph histories (tests/graph_history_oracle.py)."""
    return lambda model, ntk, rck, rows, cols: GraphHistoryOracle(model, ntk, rck, rows=rows, cols=cols)


@pytest.fixture
def gh_network_factory():
    return lambda model, ntk, rck, tk, rf: GraphHistoryOracle(model, ntk, rck, tk, rf)


def _status(ei):
    return ei.value.status


def _lattice(factory, model="izh", graph="grid", stdp=True, seed=3, rows=7, cols=9, bcm=False, history=False):
    lat = SC.build_lattice(factory, model=model, rows=rows, cols=cols, seed=seed, graph=graph, stdp=stdp, history=history)
    if bcm:
        lat.plasticity = S.BCM(decay=0.05, average_scalar=0.5, dt=1e-6)
    return lat


def _stepwise_weights(lat, n):
    """The weights get_graph_csr reports after each of n run(1) calls."""
    out = []
    for _ in range(n):
        lat.run_lattice(1)
        out.append(lat.graph_csr()[2].copy())
    return np.array(out, f32).reshape(n, -1)


def _network_stepwise(net, pairs, n):
    """Per block: the weights before each of n run(1) calls (what LatticeNetwork's record k holds)."""
    out = {p: [] for p in pairs}
    for _ in range(n):
        for p in pairs:
            out[p].append(net._be.get_connection_csr(*p)[2].copy())
        net.run_lattices(1)
    return {p: np.array(v, f32).reshape(n, -1) for p, v in out.items()}


NET_PAIRS = ((0, 1), (1, 2), (2, 1), (1, 1))


def _net(lattice_factory, network_factory, **kw):
    net = build_network(lattice_factory, network_factory, train="rate", **kw)
    net.get_lattice(1).update_graph_history = True
    net.update_connecting_graph_history = True
    return net


# ------------------------------------------------------------------ CPU tier: oracle through the front end
@pytest.mark.parametrize("graph", ["grid", "csr"])
@pytest.mark.parametrize("model", ["izh", "lif"])
def test_lattice_stdp_history_is_the_weights_after_each_step(model, graph, gh_lattice_factory):
    a, b = _lattice(gh_lattice_factory, model, graph), _lattice(gh_lattice_factory, model, graph)
    a.update_graph_history = True
    a.run_lattice(80)
    h = a.graph_history.history
    want = _stepwise_weights(b, 80)
    assert h.dtype == np.float32 and h.shape == want.shape
    assert (h == want).all()
    assert np.abs(h[-1] - h[0]).max() > 0, "STDP must move the weights for this to be a test"
    assert (a.graph_csr()[2] == h[-1]).all()


def test_network_stdp_history_is_the_weights_each_step_read(gh_lattice_factory, gh_network_factory):
    a = _net(gh_lattice_factory, gh_network_factory)
    b = _net(gh_lattice_factory, gh_network_factory)
    w0 = {p: a._be.get_connection_csr(*p)[2].copy() for p in NET_PAIRS}
    a.run_lattices(30)
    want = _network_stepwise(b, NET_PAIRS, 30)
    for p in NET_PAIRS:
        h = (a.get_lattice(1).graph_history if p == (1, 1) else a.connecting_graph_history(*p)).history
        assert h.shape == want[p].shape, p
        assert (h == want[p]).all(), p
        assert (h[0] == w0[p]).all(), p
    assert np.abs(a.connecting_graph_history(0, 1).history[-1] - w0[(0, 1)]).max() > 0
    # lattice 2 did not ask for its own graph (it has none): nothing is kept for it
    assert a._be.graph_history(2, 2).shape == (0, 0)


def test_bcm_lattice_history(gh_lattice_factory):
    a = _lattice(gh_lattice_factory, "bcm_izh", "random", bcm=True, rows=4, cols=5, seed=6)
    b = _lattice(gh_lattice_factory, "bcm_izh", "random", bcm=True, rows=4, cols=5, seed=6)
    a.update_graph_history = True
    a.run_lattice(60)
    want = _stepwise_weights(b, 60)
    assert (a.graph_history.history == want).all()
    assert np.abs(want[-1] - want[0]).max() > 0


def test_static_weights_are_recorded_every_step(gh_lattice_factory):
    a = _lattice(gh_lattice_factory, "izh", "csr", stdp=False)
    a.update_graph_history = True
    a.run_lattice(12)
    h = a.graph_history.history
    assert h.shape == (12, a.graph_csr()[2].size)
    assert (h == a.graph_csr()[2][None, :]).all()


def test_split_runs_and_reset(gh_lattice_factory):
    a, b = _lattice(gh_lattice_factory), _lattice(gh_lattice_factory)
    a.update_graph_history = b.update_graph_history = True
    a.run_lattice(3)
    a.run_lattice(4)
    b.run_lattice(7)
    assert (a.graph_history.history == b.graph_history.history).all() and a.graph_history.history.shape[0] == 7
    a.reset_timing()   # reset_timing keeps the records
    assert a.graph_history.history.shape[0] == 7
    a.graph_history.reset()
    assert a.graph_history.history.shape[0] == 0


def test_adjacency_is_frozen_while_records_exist(gh_lattice_factory):
    a = _lattice(gh_lattice_factory)
    a.update_graph_history = True
    a.run_lattice(5)
    a.edit_weight((0, 0), (0, 1), 0.25)   # an existing edge: allowed
    with pytest.raises(ERRORS) as ei:
        a.edit_weight((0, 0), (4, 5), 1.0)   # a new edge
    assert _status(ei) == K.SNN_UNSUPPORTED
    with pytest.raises(ERRORS) as ei:
        a.connect_grid(2, 1.0)
    assert _status(ei) == K.SNN_UNSUPPORTED
    a.graph_history.reset()
    a.edit_weight((0, 0), (4, 5), 1.0)
    assert a.get_weight((0, 0), (4, 5)) == 1.0


def test_dense_matches_get_graph_dense(gh_lattice_factory):
    a, b = _lattice(gh_lattice_factory, graph="csr"), _lattice(gh_lattice_factory, graph="csr")
    a.update_graph_history = True
    a.run_lattice(9)
    for step in range(9):
        b.run_lattice(1)
        c, w = a.graph_history.dense(step)
        cb, wb = b.graph_dense()
        assert (c == cb).all() and (w == wb).all()
    rp, pre, _ = a.graph_csr()
    assert (a.graph_history.row_ptr == rp).all() and (a.graph_history.pre == pre).all()


def test_reward_modulated_lattice_refuses_graph_history(gh_lattice_factory):
    lat = _lattice(gh_lattice_factory, graph="random")
    r = SC.build_lattice(gh_lattice_factory, model="izh", rows=3, cols=4, seed=5, graph="random", cls=S.RewardModulatedLattice)
    r.update_graph_history = True
    with pytest.raises(ERRORS) as ei:
        r.run_lattice(2)
    assert _status(ei) == K.SNN_UNSUPPORTED
    assert lat.update_graph_history is False and r.internal_clock == 0


# ------------------------------------------------------------------ GPU tier
@pytest.fixture(params=["auto", "tma", "tma_l1"])
def kernel_path(request, monkeypatch):
    """The automatic kernel choice, the TMA-staged kernels forced where eligible, and the window kernel off (as in
    tests/test_gpu_parity.py)."""
    monkeypatch.setenv("SNN_B200_TMA", "1" if request.param == "auto" else "2")
    monkeypatch.setenv("SNN_B200_WIN", "0" if request.param == "tma_l1" else "1")
    return request.param


@pytest.mark.gpu
@pytest.mark.parametrize("graph", ["grid", "grid2", "csr"])
@pytest.mark.parametrize("model", ["izh", "lif"])
def test_device_matches_oracle_in_segments(model, graph, kernel_path, gh_lattice_factory):
    """STDP, segment by segment from identical state (spiking lattices are chaotic, see scenarios.lockstep_lattices): the
    records at rtol 1e-4 (STDP calls expf), the rasters exactly."""
    kw = dict(model=model, rows=7, cols=9, seed=3, graph=graph, stdp=True, history=True)
    a, b = SC.build_lattice(None, **kw), SC.build_lattice(gh_lattice_factory, **kw)
    for L in (a, b):
        # weaker than the default a = 2, whose unbounded weights run away within a few hundred steps (plasticity/mod.rs:64)
        L.plasticity = S.STDP(a_plus=0.05, a_minus=0.05)
        L.update_graph_history = True
    moved = 0.0
    for seg in range(8):
        a.run_lattice(25)
        b.run_lattice(25)
        ha, hb = a.graph_history.history, b.graph_history.history
        assert ha.shape == hb.shape == (25, b.graph_csr()[2].size)
        np.testing.assert_allclose(ha, hb, rtol=1e-4, atol=1e-5, err_msg=f"graph records of segment {seg}")
        assert (a.spike_history.history == b.spike_history.history).all(), f"raster of segment {seg}"
        SC.assert_close_robust(a.grid_history.history, b.grid_history.history, 1e-4, 1e-3, f"segment {seg}")
        moved = max(moved, float(np.abs(hb[-1] - hb[0]).max()))
        for L in (a, b):
            L.graph_history.reset()   # also clears the grid / spike records, and frees the adjacency for the re-sync
        SC.copy_lattice_state(b, a, weights=True)
    assert moved > 0


@pytest.mark.gpu
@pytest.mark.parametrize("graph", ["grid", "random"])
def test_bcm_history_bit_exact(graph, gh_lattice_factory):
    kw = dict(model="bcm_izh", rows=7, cols=9, seed=4, graph=graph, stdp=True)
    a, b = SC.build_lattice(None, **kw), SC.build_lattice(gh_lattice_factory, **kw)
    for L in (a, b):
        L.plasticity = S.BCM(decay=0.05, average_scalar=0.5, dt=1e-6)
        L.update_graph_history = True
        L.run_lattice(150)
        L.run_lattice(100)
    ha, hb = a.graph_history.history, b.graph_history.history
    assert ha.shape == hb.shape == (250, b.graph_csr()[2].size)
    assert (ha == hb).all()
    assert np.abs(hb[-1] - hb[0]).max() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("graph", ["grid", "csr"])
def test_device_lattice_history_equals_stepwise_reads(graph, kernel_path):
    a, b = _lattice(None, "izh", graph, rows=20, cols=24), _lattice(None, "izh", graph, rows=20, cols=24)
    a.update_graph_history = True
    a.run_lattice(25)
    a.run_lattice(15)
    h = a.graph_history.history
    want = _stepwise_weights(b, 40)
    assert h.shape == want.shape and (h == want).all()
    assert np.abs(want[-1] - want[0]).max() > 0


@pytest.mark.gpu
def test_device_network_history_equals_stepwise_reads():
    """72 spike trains feed lattice 1 all-to-all (the wide-row kernel), STDP on the connecting blocks and lattice 1's graph."""
    a, b = _net(None, None, st_shape=(8, 9)), _net(None, None, st_shape=(8, 9))
    a.run_lattices(20)
    a.run_lattices(15)
    want = _network_stepwise(b, NET_PAIRS, 35)
    for p in NET_PAIRS:
        h = (a.get_lattice(1).graph_history if p == (1, 1) else a.connecting_graph_history(*p)).history
        assert h.shape == want[p].shape and (h == want[p]).all(), p
    assert np.abs(want[(0, 1)][-1] - want[(0, 1)][0]).max() > 0


def _state(lat, last):
    return lat.get_field("current_voltage").copy(), lat.spike_history.history[-last:].copy(), lat.graph_csr()[2].copy()


@pytest.mark.gpu
@pytest.mark.parametrize("graph", ["grid", "csr"])
@pytest.mark.parametrize("stdp", [True, False])
def test_recording_does_not_perturb_the_run(graph, stdp, kernel_path):
    kw = dict(model="izh", rows=40, cols=50, seed=9, graph=graph, stdp=stdp, history=True)
    on, off, never = SC.build_lattice(None, **kw), SC.build_lattice(None, **kw), SC.build_lattice(None, **kw)
    on.update_graph_history = True
    on.run_lattice(60)
    off.update_graph_history = True
    off.run_lattice(1)
    off.update_graph_history = False
    off.graph_history.reset()   # (clears the grid and spike records too: the last 59 steps are compared)
    off.run_lattice(59)
    never.run_lattice(60)
    assert on.graph_history.history.shape[0] == 60 and off.graph_history.history.shape[0] == 0
    for x, last in ((on, 60), (off, 59)):
        for u, v in zip(_state(x, last), _state(never, last)):
            assert (u == v).all()
    # with the flag off again the run is the same launch for launch as a handle that never set it
    off._push_options(); never._push_options()
    assert off._be.run_timed(30)[1] == never._be.run_timed(30)[1]


@pytest.mark.gpu
def test_network_recording_does_not_perturb_the_run():
    on, never = _net(None, None), build_network(None, None, train="rate")
    on.run_lattices(50)
    never.run_lattices(50)
    for lid in (1, 2):
        assert (on.get_lattice(lid).grid_history.history == never.get_lattice(lid).grid_history.history).all()
        assert (on.get_lattice(lid).spike_history.history == never.get_lattice(lid).spike_history.history).all()
    for p in NET_PAIRS:
        assert (on._be.get_connection_csr(*p)[2] == never._be.get_connection_csr(*p)[2]).all()


@pytest.mark.gpu
def test_refused_configurations_leave_the_state_unchanged():
    from snn_b200.backend import CudaLatticeBackend
    # a row strip of a partitioned lattice
    be = CudaLatticeBackend(K.MODEL_IZH, rows=8, cols=8, rank=0, world=2)
    be.connect_grid(0, 1, 1.0)
    be.set_option(K.OPT_UPDATE_GRAPH_HISTORY, 1)
    with pytest.raises(S.SnnError) as ei:
        be.run(3)
    assert _status(ei) == K.SNN_UNSUPPORTED and be.get_option(K.OPT_INTERNAL_CLOCK) == 0
    be.close()
    # a reward-modulated lattice
    r = SC.build_lattice(None, model="izh", rows=6, cols=7, seed=5, graph="random", cls=S.RewardModulatedLattice)
    v0, w0 = r.get_field("current_voltage").copy(), r.graph_csr()[2].copy()
    r.update_graph_history = True
    with pytest.raises(S.SnnError) as ei:
        r.run_lattice(3)
    assert _status(ei) == K.SNN_UNSUPPORTED
    with pytest.raises(S.SnnError) as ei:
        r.run_lattice_with_rewards([1.0, 0.5])
    assert _status(ei) == K.SNN_UNSUPPORTED
    assert r.internal_clock == 0 and (r.get_field("current_voltage") == v0).all() and (r.graph_csr()[2] == w0).all()
    assert r._be.graph_history().shape == (0, 0)


@pytest.mark.gpu
def test_device_adjacency_frozen_and_dense():
    a = _lattice(None, graph="csr")
    a.update_graph_history = True
    a.run_lattice(6)
    a.edit_weight((0, 0), (0, 1), 0.25)
    with pytest.raises(S.SnnError) as ei:
        a.edit_weight((0, 0), (4, 5), 1.0)
    assert _status(ei) == K.SNN_UNSUPPORTED
    c, w = a.graph_history.dense(5)
    cd, _ = a.graph_dense()
    assert (c == cd).all() and (w[c == 1] != 0).any()
    a.graph_history.reset()
    a.edit_weight((0, 0), (4, 5), 1.0)
    assert a.get_weight((0, 0), (4, 5)) == 1.0
