"""Parity of the CUDA path (through the C ABI) against the CPU oracle and the golden fixtures.

Bar (BASELINE.json north_star / SURVEY.md §8c): adjacency and spike rasters bit-exact for the deterministic
models; state within rel. 1e-4 for models that call expf/powf; Poisson runs by firing statistics.
"""
import numpy as np
import pytest

import golden_util as G
import scenarios as SC
import snn_b200 as S
from snn_b200 import _capi as K

pytestmark = pytest.mark.gpu
f32 = np.float32


@pytest.fixture(autouse=True, params=["auto", "tma", "tma_l1"])
def kernel_path(request, monkeypatch):
    """Every parity test runs three times: with the automatic kernel choice (for small lattices the cooperative multi-step
    step_multi_kernel, in its 16-CTA cluster variant up to 320 slices), with
    the TMA-staged persistent kernels forced wherever they are eligible (stencil graphs: the window-staged step_win_kernel
    for radius 1, the L1-gather step_tma_kernel for larger radii), and with the window kernel disabled so that
    step_tma_kernel also serves radius 1 — all three are held to the same bar."""
    monkeypatch.setenv("SNN_B200_TMA", "1" if request.param == "auto" else "2")
    monkeypatch.setenv("SNN_B200_WIN", "0" if request.param == "tma_l1" else "1")
    return request.param


def pair(oracle_factory, **kw):
    return SC.build_lattice(None, **kw), SC.build_lattice(oracle_factory, **kw)


def state_fields(model):
    return list(SC.MODELS[model]().scalar_fields())


# ------------------------------------------------------------------ golden fixtures
@pytest.mark.parametrize("name", G.NAMES)
def test_cuda_matches_golden(name):
    from snn_b200.backend import CudaLatticeBackend
    g = G.load(name)
    be = G.replay(g, lambda m, n, r, rows, cols: CudaLatticeBackend(m, n, r, rows, cols))
    G.check(name, be, g)


# ------------------------------------------------------------------ deterministic models: bit exact
@pytest.mark.parametrize("graph", ["grid", "grid2", "random", "csr", "all", "none"])
@pytest.mark.parametrize("model", SC.EXACT_MODELS)
def test_electrical_bit_exact(model, graph, oracle_lattice_factory):
    a, b = pair(oracle_lattice_factory, model=model, rows=7, cols=9, seed=3, graph=graph)
    a.run_lattice(500)
    b.run_lattice(500)
    assert b.spike_history.history.sum() > 0, "scenario must spike to be a meaningful raster test"
    SC.compare_lattices(a, b, exact=True, fields=state_fields(model))
    ca, wa = a.graph_dense()
    cb, wb = b.graph_dense()
    assert (ca == cb).all() and (wa == wb).all()


@pytest.mark.parametrize("shape", [(1, 1), (1, 33), (33, 1), (5, 13), (32, 32), (31, 33)])
def test_ragged_shapes_bit_exact(shape, oracle_lattice_factory):
    a, b = pair(oracle_lattice_factory, model="izh", rows=shape[0], cols=shape[1], seed=5, graph="grid")
    a.run_lattice(300)
    b.run_lattice(300)
    SC.compare_lattices(a, b, exact=True, fields=state_fields("izh"))


def test_config1_izhikevich_100x100_first_steps(oracle_lattice_factory):
    """BASELINE.json configs[0]: Izhikevich 100x100, electrical, 8-neighbour grid, dt=0.1 (raster bit-exact)."""
    a, b = pair(oracle_lattice_factory, model="izh", rows=100, cols=100, seed=11, graph="grid", hetero=False, c_m=5.0)
    a.run_lattice(1000)
    b.run_lattice(1000)
    assert b.spike_history.history.sum() > 100
    SC.compare_lattices(a, b, exact=True, fields=state_fields("izh"))


# ------------------------------------------------------------------ reduced histories (SURVEY 8a19)
@pytest.mark.parametrize("kind", ["average", "eeg"])
@pytest.mark.parametrize("shape", [(7, 9), (40, 50)])
def test_average_and_eeg_history(kind, shape, oracle_lattice_factory):
    """AverageVoltageHistory / EEGHistory (neuron/mod.rs:231-322).  The reference sums sequentially in f32; the device
    reduces the same voltages in f64 in a fixed order, so the bar is the rounding of a length-N f32 sum: rel 1e-5, and
    1e-6 against the f64 mean of the (bit-exact) grid voltages."""
    ht = S.AverageVoltageHistory if kind == "average" else S.EEGHistory
    kw = dict(model="izh", rows=shape[0], cols=shape[1], seed=3, graph="grid")
    a, b = SC.build_lattice(None, history_type=ht, **kw), SC.build_lattice(oracle_lattice_factory, history_type=ht, **kw)
    g = SC.build_lattice(None, **kw)   # same lattice recording the full grid
    if kind == "eeg":
        for L in (a, b):
            L.grid_history.reference_voltage, L.grid_history.distance, L.grid_history.conductivity = 0.5, 1.25, 100.0
    for L in (a, b, g):
        L.run_lattice(120)
        L.run_lattice(80)   # histories append across run calls
    ha, hb = a.grid_history.history, b.grid_history.history
    assert ha.shape == hb.shape == (200,) and ha.dtype == np.float32
    np.testing.assert_allclose(ha, hb, rtol=1e-5, atol=1e-5)
    v = g.grid_history.history.reshape(200, -1)
    if kind == "average":
        np.testing.assert_allclose(ha, v.astype(np.float64).mean(axis=1), rtol=1e-6, atol=1e-6)
    else:
        tot = (v - f32(0.5)).astype(np.float64).sum(axis=1)
        np.testing.assert_allclose(ha, tot / (4 * np.pi * 100.0 * 1.25), rtol=1e-6, atol=1e-6)
    assert (a.spike_history.history == b.spike_history.history).all()
    a.grid_history.reset()
    assert a.grid_history.history.shape == (0,)


# ------------------------------------------------------------------ BCM plasticity (SURVEY 8f rank 4)
@pytest.mark.parametrize("graph", ["grid", "random"])
def test_bcm_plasticity_bit_exact(graph, oracle_lattice_factory):
    """Lattice<BCMIzhikevichNeuron, ..., BCM, ...> (plasticity/mod.rs:80-112): no transcendental anywhere, so voltages, rasters,
    activities and weights must match the oracle bit for bit."""
    kw = dict(model="bcm_izh", rows=7, cols=9, seed=4, graph=graph, stdp=True)
    a, b = SC.build_lattice(None, **kw), SC.build_lattice(oracle_lattice_factory, **kw)
    for L in (a, b):
        L.plasticity = S.BCM(decay=0.05, average_scalar=0.5, dt=1e-6)   # tame: activities grow with the never-reset num_spikes
    w0 = b.graph_csr()[2].copy()
    for L in (a, b):
        L.run_lattice(250)
        L.run_lattice(150)
    assert b.spike_history.history.sum() > 20
    SC.compare_lattices(a, b, exact=True, fields=state_fields("bcm_izh"))
    (rpa, pa, wa), (rpb, pb, wb) = a.graph_csr(), b.graph_csr()
    assert (pa == pb).all() and (wa == wb).all()
    assert np.abs(wb - w0).max() > 1e-5 and np.isfinite(wb).all(), "the BCM rule must have moved the weights"
    a.do_plasticity = b.do_plasticity = False
    a.run_lattice(20)
    assert (a.graph_csr()[2] == wa).all()


# ------------------------------------------------------------------ reward-modulated lattices (SURVEY 8f rank 1)
@pytest.mark.parametrize("canonical", [True, False])
@pytest.mark.parametrize("graph,shape", [("grid", (9, 11)), ("random", (6, 7)), ("grid", (300, 300))])
def test_reward_modulated_lattice(graph, shape, canonical, oracle_lattice_factory):
    """RewardModulatedLattice with RewardModulatedSTDP over TraceRSTDP weights (neuron/mod.rs:2717-3416, plasticity/mod.rs:114-234):
    every edge is updated twice per step from the ping-ponged last_firing_time.  Lock-step segments against the oracle (the
    weights feed back into a chaotic lattice): rasters bit-exact, voltages / weights / traces to expf rounding."""
    big = shape[0] * shape[1] > 10000
    kw = dict(model="izh", rows=shape[0], cols=shape[1], seed=9, graph=graph, cls=S.RewardModulatedLattice, history=not big)
    a, b = SC.build_lattice(None, **kw), SC.build_lattice(oracle_lattice_factory, **kw)
    for L in (a, b):
        L.reward_modulator = S.RewardModulatedSTDP(tau_c=0.05, a_plus=0.1, a_minus=0.08)   # tame: the rule has no weight clamp
    rng = np.random.default_rng(1)
    w0 = b.graph_csr()[2].copy()
    if not canonical:
        # traces stored through edit_weight with an odd call phase: leaves the device kernel's counter == 0 / dw == 0 fast path
        cnt0 = (rng.random(w0.size) < 0.5).astype(np.uint32)
        dw0 = (rng.uniform(-0.01, 0.01, w0.size) * cnt0).astype(f32)
        c0 = rng.uniform(-0.001, 0.001, w0.size).astype(f32)
        for L in (a, b):
            L.set_graph_traces(None, cnt0, dw0, c0)
    # the lattice is strongly chaotic (measured: an ulp-level weight difference grows to 0.4 mV within 40 free-running steps)
    total, seg, done = (40, 10, 0) if big else (150, 10, 0)
    while done < total:
        rewards = rng.uniform(-0.3, 0.3, seg).astype(f32)
        for L in (a, b):
            if (done // seg) % 3 == 2:
                L.run_lattice(seg)                 # RunLattice::run_lattice: no reward signal, modulation still on
            else:
                L.run_lattice_with_rewards(rewards)
        if not big:
            ha, hb = a.grid_history.history[done:done + seg], b.grid_history.history[done:done + seg]
            SC.assert_close_robust(ha, hb, 1e-4, 1e-3, f"segment at {done}")
            assert (a.spike_history.history[done:done + seg] == b.spike_history.history[done:done + seg]).all()
        assert (a.get_field("last_firing_time") == b.get_field("last_firing_time")).all()
        (rpa, pa, wa), (rpb, pb, wb) = a.graph_csr(), b.graph_csr()
        assert (rpa == rpb).all() and (pa == pb).all()
        np.testing.assert_allclose(wa, wb, rtol=1e-4, atol=1e-5, err_msg=f"weights after step {done + seg}")
        (ca, da, cca), (cb, db, ccb) = a.graph_traces(), b.graph_traces()
        assert (ca == cb).all()
        np.testing.assert_allclose(da, db, rtol=1e-4, atol=1e-6)
        np.testing.assert_allclose(cca, ccb, rtol=1e-4, atol=1e-6)
        assert a.reward_modulator.dopamine == pytest.approx(b.reward_modulator.dopamine, rel=1e-5)
        SC.copy_lattice_state(b, a, weights=False)   # re-synchronise the neurons (see scenarios.lockstep_lattices) ...
        a.set_graph_traces(wb, cb, db, ccb)          # ... and the TraceRSTDP values, in place
        done += seg
    assert (b.get_field("last_firing_time") >= 0).sum() > 5
    assert np.abs(b.graph_csr()[2] - w0).max() > 1e-3, "the modulator must have moved the weights"
    a.do_modulation = b.do_modulation = False
    wa0 = a.graph_csr()[2].copy()
    a.run_lattice(10)
    assert (a.graph_csr()[2] == wa0).all(), "do_modulation = false freezes the weights"


# ------------------------------------------------------------------ transcendental models: tolerance
@pytest.mark.parametrize("model,graph,steps", [("adex", "grid", 500), ("adex", "random", 500), ("hh", "grid", 2000),
                                               ("hh", "random", 2000)])
def test_electrical_tolerance_models(model, graph, steps, oracle_lattice_factory):
    a, b = pair(oracle_lattice_factory, model=model, rows=6, cols=7, seed=4, graph=graph, gap=SC.drive_current(model))
    a.run_lattice(steps)
    b.run_lattice(steps)
    ha, hb = a.grid_history.history, b.grid_history.history
    np.testing.assert_allclose(ha[:100], hb[:100], rtol=1e-4, atol=1e-3)
    assert np.abs(ha - hb).max() <= 2.0  # tests/gpu_accuracy.rs:73
    assert G.raster_close(a.spike_history.history.reshape(steps, -1), b.spike_history.history.reshape(steps, -1))


# ------------------------------------------------------------------ chemical synapses
@pytest.mark.parametrize("electrical", [True, False])
@pytest.mark.parametrize("graph", ["grid", "random"])
def test_chemical_approximate_ampa_bit_exact(graph, electrical, oracle_lattice_factory):
    """Izhikevich + ApproximateNeurotransmitter/ApproximateReceptor AMPA: no transcendental -> exact."""
    a, b = pair(oracle_lattice_factory, model="izh", rows=6, cols=8, seed=7, graph=graph, chem="approx_ampa",
                electrical=electrical)
    a.run_lattice(600)
    b.run_lattice(600)
    assert b.spike_history.history.sum() > 0
    SC.compare_lattices(a, b, exact=True, fields=state_fields("izh") + [
        "neurotransmitters$t", "receptors$AMPA$r$kinetics$r", "receptors$AMPA_current"])


@pytest.mark.parametrize("model,chem,steps", [("izh", "approx_all", 400), ("lif", "expdecay_all", 400), ("qif", "discrete_ampa", 400),
                                              ("hh", "destexhe_all", 2000), ("izh", "destexhe_all", 400)])
def test_chemical_tolerance(model, chem, steps, oracle_lattice_factory):
    a, b = pair(oracle_lattice_factory, model=model, rows=5, cols=6, seed=8, graph="grid", chem=chem,
                gap=SC.drive_current(model), c_m=(20.0 if model == "izh" else None))
    a.run_lattice(steps)
    b.run_lattice(steps)
    ha, hb = a.grid_history.history, b.grid_history.history
    np.testing.assert_allclose(ha[:50], hb[:50], rtol=1e-4, atol=1e-3)
    assert np.abs(ha - hb).max() <= 5.0  # tests/gpu_accuracy.rs:163
    assert G.raster_close(a.spike_history.history.reshape(steps, -1), b.spike_history.history.reshape(steps, -1))
    for ty in ("AMPA",) if chem.endswith("ampa") else ("AMPA", "NMDA", "GABA"):
        np.testing.assert_allclose(a.get_field(f"receptors${ty}$r$kinetics$r"), b.get_field(f"receptors${ty}$r$kinetics$r"),
                                   rtol=1e-3, atol=1e-4)


def test_heterogeneous_neurotransmitter_types(oracle_lattice_factory):
    """Per-neuron type sets: the per-type averaging denominator counts only presynaptic neurons that have the type
    (iterate_and_spike/mod.rs:2852-2863); inhibition is a negative weight (SURVEY appendix A.11)."""
    lat = []
    for fac in (None, oracle_lattice_factory):
        L = SC.build_lattice(fac, model="izh", rows=5, cols=5, seed=9, graph="random", chem="approx_all")
        rng = np.random.default_rng(3)
        L.set_field("neurotransmitters$flags", (rng.random((25, 3)) < 0.6).astype(np.uint32))
        L.set_field("receptors$flags", (rng.random((25, 3)) < 0.7).astype(np.uint32))
        c, w = L.graph_dense()
        w = w * np.where(rng.random(w.shape) < 0.3, -1.0, 1.0).astype(f32)
        L._be.connect_dense(L._bid, L._bid, c, w)
        lat.append(L)
    a, b = lat
    a.run_lattice(300)
    b.run_lattice(300)
    ha, hb = a.grid_history.history, b.grid_history.history
    np.testing.assert_allclose(ha[:50], hb[:50], rtol=1e-4, atol=1e-3)
    assert np.abs(ha - hb).max() <= 5.0
    assert (a.get_field("neurotransmitters$flags") == b.get_field("neurotransmitters$flags")).all()


# ------------------------------------------------------------------ STDP
@pytest.mark.parametrize("model,graph", [("izh", "grid"), ("izh", "random"), ("lif", "grid"), ("lif", "all")])
def test_stdp_weights(model, graph, oracle_lattice_factory):
    """Short horizon from identical state: weights to 1e-5 (expf), raster exact."""
    a, b = pair(oracle_lattice_factory, model=model, rows=6, cols=6, seed=12, graph=graph, stdp=True,
                c_m=(10.0 if model == "izh" else None))
    for L in (a, b):
        L.plasticity = S.STDP(a_plus=0.05, a_minus=0.04, tau_plus=4.5, tau_minus=3.0, dt=0.1)
    w0 = b.graph_dense()[1].copy()
    a.run_lattice(300)
    b.run_lattice(300)
    assert b.spike_history.history.sum() > 10
    (ca, wa), (cb, wb) = a.graph_dense(), b.graph_dense()
    assert (ca == cb).all()
    assert np.abs(wb - w0).max() > 0.01
    np.testing.assert_allclose(wa, wb, rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(a.grid_history.history, b.grid_history.history, rtol=1e-4, atol=1e-3)
    assert (a.spike_history.history == b.spike_history.history).all()


@pytest.mark.parametrize("model,graph,chem", [("izh", "grid", None), ("izh", "random", "approx_all"), ("lif", "grid", "approx_ampa"),
                                              ("hh", "grid", "destexhe_all")])
def test_stdp_long_horizon_lockstep(model, graph, chem, oracle_lattice_factory):
    """Default-strength STDP (a = 2) over 600 steps, compared segment by segment (see scenarios.lockstep_lattices)."""
    a, b = pair(oracle_lattice_factory, model=model, rows=6, cols=7, seed=14, graph=graph, stdp=True, chem=chem,
                gap=SC.drive_current(model))
    spikes = SC.lockstep_lattices(a, b, 600 if model != "hh" else 1500, 25, weights=True)
    assert spikes > 10


def test_stdp_run_continuity(oracle_lattice_factory):
    """Two run calls == one run call: the lazily applied last-step STDP is flushed at every API boundary and the
    clock / last_firing_time persist (SURVEY §5 checkpoint/resume)."""
    one = SC.build_lattice(None, model="izh", rows=6, cols=6, seed=13, graph="grid", stdp=True, history=False)
    two = SC.build_lattice(None, model="izh", rows=6, cols=6, seed=13, graph="grid", stdp=True, history=False)
    one.run_lattice(400)
    two.run_lattice(137)
    w_mid = two.graph_dense()[1].copy()
    two.run_lattice(263)
    assert one.internal_clock == two.internal_clock == 400
    assert (one.graph_dense()[1] == two.graph_dense()[1]).all()
    assert (one.get_field("current_voltage") == two.get_field("current_voltage")).all()
    assert (one.get_field("last_firing_time") == two.get_field("last_firing_time")).all()
    ref = SC.build_lattice(oracle_lattice_factory, model="izh", rows=6, cols=6, seed=13, graph="grid", stdp=True, history=False)
    ref.run_lattice(137)
    np.testing.assert_allclose(w_mid, ref.graph_dense()[1], rtol=1e-4, atol=1e-5)


# ------------------------------------------------------------------ networks
def build_network(lattice_factory, network_factory, train="rate", stdp=True, chemical=True, electrical=True, seed=21,
                  st_shape=(3, 4), refract=None):
    """MNIST-shaped miniature of BASELINE.json configs[3]: spike trains -> excitatory <-> inhibitory."""
    rng = np.random.default_rng(seed)
    T = S.IonotropicNeurotransmitterType
    exc_base = S.IzhikevichNeuron(gap_conductance=5.0, c_m=10.0)
    exc_base.synaptic_neurotransmitters[T.AMPA] = S.ApproximateNeurotransmitter()
    exc_base.receptors[T.AMPA] = S.AMPAReceptor()
    exc_base.receptors[T.GABA] = S.GABAReceptor()
    inh_base = exc_base.clone()
    inh_base.synaptic_neurotransmitters = {T.GABA: S.ApproximateNeurotransmitter(clearance_constant=0.02)}
    exc = S.Lattice(S.IzhikevichNeuron, id=1, backend_factory=lattice_factory)
    exc.populate(exc_base, 4, 5)
    inh = S.Lattice(S.IzhikevichNeuron, id=2, backend_factory=lattice_factory)
    inh.populate(inh_base, 4, 5)
    for L in (exc, inh):
        L.set_field("current_voltage", rng.uniform(-65, 20, 20).astype(f32))
        L.set_field("b", rng.uniform(0.25, 0.33, 20).astype(f32))
        L.update_grid_history = L.update_spike_history = True
        L.do_plasticity = stdp
        L.plasticity = S.STDP(a_plus=0.03, a_minus=0.03)
    exc.connect(lambda x, y: x != y and abs(x[0] - y[0]) + abs(x[1] - y[1]) <= 1, lambda x, y: 0.5)
    if train == "rate":
        st_cls, base = S.RateSpikeTrain, S.RateSpikeTrain(rate=2.0)
    elif train == "poisson":
        st_cls, base = S.PoissonNeuron, S.PoissonNeuron.from_firing_rate(200.0, 0.1)
    else:
        st_cls, base = S.PresetSpikeTrain, S.PresetSpikeTrain(firing_times=[1.0, 2.5, 0.7])
    base.synaptic_neurotransmitters[T.AMPA] = S.ApproximateNeurotransmitter()
    if refract is not None:
        base.neural_refractoriness = refract
    st = S.SpikeTrainLattice(st_cls, id=0, network_backend_factory=network_factory)
    n_st = st_shape[0] * st_shape[1]
    st.populate(base, *st_shape)
    if train == "rate":
        st.set_field("rate", rng.choice([0.0, 1.5, 2.0, 3.0], n_st).astype(f32))
    st.update_spike_history = True
    net = S.LatticeNetwork.generate_network([exc, inh], [st], backend_factory=network_factory)
    wmat = rng.uniform(0, 1, (n_st, 20)).astype(f32)
    net.connect(0, 1, lambda x, y: True, lambda x, y: float(wmat[x[0] * st_shape[1] + x[1], y[0] * 5 + y[1]]))
    net.connect(1, 2, lambda x, y: x == y, lambda x, y: 1.0)
    net.connect(2, 1, lambda x, y: x != y, lambda x, y: -1.0)
    net.electrical_synapse, net.chemical_synapse = electrical, chemical
    return net


PAIRS = ((0, 1), (1, 2), (2, 1), (1, 1))


def _sync_network(src, dst):
    for lid in (1, 2):
        SC.copy_lattice_state(src.get_lattice(lid), dst.get_lattice(lid), weights=False)
    SC.copy_lattice_state(src.get_spike_train_lattice(0), dst.get_spike_train_lattice(0), weights=False)
    for pre, post in PAIRS:
        c, w = src._be.get_connection_dense(pre, post)
        dst._be.connect_dense(pre, post, c, w)


@pytest.mark.parametrize("st_shape", [(3, 4), (8, 9)])
@pytest.mark.parametrize("train", ["rate", "preset"])
@pytest.mark.parametrize("mode", [(True, True), (True, False), (False, True)])
def test_network_deterministic_trains(train, mode, st_shape, oracle_lattice_factory, oracle_network_factory):
    """Spike trains -> excitatory <-> inhibitory with STDP on every lattice, compared in lock-step segments (the
    network is chaotic; see scenarios.lockstep_lattices).  With 72 spike trains the mean slice width passes
    kWideMinWidth and the wide-row kernel (step_wide.cu) steps the network."""
    a = build_network(None, None, train=train, electrical=mode[0], chemical=mode[1], st_shape=st_shape)
    b = build_network(oracle_lattice_factory, oracle_network_factory, train=train, electrical=mode[0], chemical=mode[1],
                      st_shape=st_shape)
    total, seg, done, spikes = 400, 20, 0, 0
    while done < total:
        a.run_lattices(seg)
        b.run_lattices(seg)
        sa = a.get_spike_train_lattice(0).spike_history.history[done:done + seg]
        sb = b.get_spike_train_lattice(0).spike_history.history[done:done + seg]
        assert (sa == sb).all()
        for lid in (1, 2):
            ha, hb = a.get_lattice(lid).grid_history.history[done:done + seg], b.get_lattice(lid).grid_history.history[done:done + seg]
            SC.assert_close_robust(ha, hb, 1e-4, 1e-3, f"lattice {lid}, segment at {done}")
            ra, rb = a.get_lattice(lid).spike_history.history[done:done + seg], b.get_lattice(lid).spike_history.history[done:done + seg]
            assert (ra == rb).all(), f"lattice {lid}: raster differs in the segment at {done}"
            spikes += int(rb.sum())
        for pre, post in PAIRS:
            (ca, wa), (cb, wb) = a._be.get_connection_dense(pre, post), b._be.get_connection_dense(pre, post)
            assert (ca == cb).all()
            np.testing.assert_allclose(wa, wb, rtol=1e-5, atol=1e-6, err_msg=f"weights {pre}->{post} after step {done + seg}")
        assert a.internal_clock == b.internal_clock == done + seg
        assert (a.get_spike_train_lattice(0).get_field("last_firing_time") == b.get_spike_train_lattice(0).get_field("last_firing_time")).all()
        _sync_network(b, a)
        done += seg
    assert spikes > 20
    w_trains = b._be.get_connection_dense(0, 1)[1]
    assert np.abs(w_trains - build_network(oracle_lattice_factory, oracle_network_factory, train=train,
                                           st_shape=st_shape)._be.get_connection_dense(0, 1)[1]).max() > 0


def test_network_electrical_rate_trains_bit_exact(oracle_lattice_factory, oracle_network_factory):
    """No plasticity, electrical only: the only transcendental is the spike-train refractoriness expf."""
    a = build_network(None, None, train="rate", stdp=False, electrical=True, chemical=False)
    b = build_network(oracle_lattice_factory, oracle_network_factory, train="rate", stdp=False, electrical=True, chemical=False)
    a.run_lattices(300)
    b.run_lattices(300)
    for lid in (1, 2):
        ha, hb = a.get_lattice(lid).grid_history.history, b.get_lattice(lid).grid_history.history
        np.testing.assert_allclose(ha, hb, rtol=1e-4, atol=1e-3)
        assert (a.get_lattice(lid).spike_history.history == b.get_lattice(lid).spike_history.history).all()


@pytest.mark.parametrize("st_shape", [(3, 4), (8, 9)])
@pytest.mark.parametrize("stdp", [False, True])
def test_network_exponential_decay_refractoriness(st_shape, stdp, oracle_lattice_factory, oracle_network_factory):
    """ExponentialDecayRefractoriness (spike_train/mod.rs:150-180) behind spike_train_gap_junction (neuron/mod.rs:119-137): the
    trains' effect on their postsynaptic neurons decays as exp(-dt_since_spike / (k / dt)) instead of the Gaussian of the
    delta-Dirac kind.  Both the narrow kernel (12 trains) and the wide-row kernel (72 trains) are covered; with STDP the
    comparison is segment-wise (expf in the weight update)."""
    kw = dict(train="rate", stdp=stdp, electrical=True, chemical=False, st_shape=st_shape)
    a = build_network(None, None, refract=S.ExponentialDecayRefractoriness(k=1.5), **kw)
    b = build_network(oracle_lattice_factory, oracle_network_factory, refract=S.ExponentialDecayRefractoriness(k=1.5), **kw)
    ref_dirac = build_network(oracle_lattice_factory, oracle_network_factory, **kw)
    assert a.get_spike_train_lattice(0)._refract == K.REFRACT_EXPONENTIAL_DECAY
    total, seg, done, spikes = 200, 25, 0, 0
    while done < total:
        a.run_lattices(seg)
        b.run_lattices(seg)
        for lid in (1, 2):
            ha, hb = a.get_lattice(lid).grid_history.history[done:done + seg], b.get_lattice(lid).grid_history.history[done:done + seg]
            np.testing.assert_allclose(ha, hb, rtol=1e-4, atol=1e-3, err_msg=f"lattice {lid}, segment at {done}")
            ra, rb = a.get_lattice(lid).spike_history.history[done:done + seg], b.get_lattice(lid).spike_history.history[done:done + seg]
            assert (ra == rb).all(), f"lattice {lid}: raster differs in the segment at {done}"
            spikes += int(rb.sum())
        _sync_network(b, a)
        done += seg
    assert spikes > 10
    # the refractoriness kind matters: the same network with the delta-Dirac kind follows another trajectory
    ref_dirac.run_lattices(total)
    assert np.abs(ref_dirac.get_lattice(1).grid_history.history - b.get_lattice(1).grid_history.history).max() > 1e-2


def test_poisson_noise_is_fresh_after_reset_timing_and_across_handles():
    """The reference draws thread_rng values on every iterate (spike_train/mod.rs:352-368): a presentation / reset_timing loop
    must not replay the same noise, and two networks built the same way must not share it (unless the caller pins the key)."""
    steps = 600
    net = build_network(None, None, train="poisson", stdp=False)
    net.run_lattices(steps)
    first = net.get_spike_train_lattice(0).spike_history.history.copy()
    net.reset_timing()
    net.get_spike_train_lattice(0).spike_history.reset()
    net.run_lattices(steps)
    second = net.get_spike_train_lattice(0).spike_history.history
    assert first.shape == second.shape and first.sum() > 20 and second.sum() > 20
    assert (first != second).any(), "reset_timing replayed the identical Poisson sequence"
    other = build_network(None, None, train="poisson", stdp=False)
    other.run_lattices(steps)
    assert (other.get_spike_train_lattice(0).spike_history.history != first).any(), "two handles share one default key"


def test_poisson_network_firing_statistics():
    """Poisson parity is statistical (reference RNG is unseeded thread_rng): the empirical rate of each train must
    sit inside a 5-sigma binomial interval around chance_of_firing, and runs must be reproducible per seed."""
    steps = 4000
    nets = [build_network(None, None, train="poisson", stdp=False) for _ in range(2)]
    for n in nets:
        n._be.set_option(K.OPT_RNG_SEED, 1234)
        n.run_lattices(steps)
    s0 = nets[0].get_spike_train_lattice(0).spike_history.history
    s1 = nets[1].get_spike_train_lattice(0).spike_history.history
    assert (s0 == s1).all()
    p = float(nets[0].get_spike_train_lattice(0).get_field("chance_of_firing")[0])
    assert p == pytest.approx(0.02, rel=1e-5)
    counts = s0.reshape(steps, -1).sum(axis=0)
    sigma = np.sqrt(steps * p * (1 - p))
    assert (np.abs(counts - steps * p) < 5 * sigma).all(), counts
    total = counts.sum()
    assert abs(total - 12 * steps * p) < 5 * np.sqrt(12) * sigma
    other = build_network(None, None, train="poisson", stdp=False)
    other._be.set_option(K.OPT_RNG_SEED, 99)
    other.run_lattices(steps)
    assert (other.get_spike_train_lattice(0).spike_history.history != s0).any()


@pytest.mark.parametrize("synapses", [(True, False), (False, True)])
def test_reference_poisson_to_izhikevich_behaviour(synapses):
    """tests/spike_train_neuron_interaction.rs:90-157 re-stated on the CUDA path."""
    T = S.IonotropicNeurotransmitterType
    iterations = 2500
    neuron = S.IzhikevichNeuron(gap_conductance=10.0)
    neuron.synaptic_neurotransmitters[T.AMPA] = S.ApproximateNeurotransmitter()
    neuron.receptors[T.AMPA] = S.AMPAReceptor()
    poisson = S.PoissonNeuron()
    poisson.synaptic_neurotransmitters[T.AMPA] = S.ApproximateNeurotransmitter()
    st = S.SpikeTrainLattice(S.PoissonNeuron, id=0)
    st.populate(poisson, 1, 1)
    lat = S.Lattice(S.IzhikevichNeuron, id=1)
    lat.populate(neuron, 1, 1)
    lat.update_spike_history = True
    net = S.LatticeNetwork.generate_network([lat], [st])
    net.connect(0, 1, lambda x, y: x == y, lambda x, y: 1.0)
    net.parallel = True
    net.electrical_synapse, net.chemical_synapse = synapses
    net.set_dt(1.0)
    net.run_lattices(iterations)
    assert net.get_lattice(1).spike_history.history.sum() <= 1
    net.get_spike_train_lattice(0).apply(lambda s: setattr(s, "chance_of_firing", (1.0 / 1.0) * 0.01))
    net.run_lattices(iterations)
    after = net.get_lattice(1).spike_history.history[iterations:].sum()
    assert after > 2, after


# ------------------------------------------------------------------ BASELINE.json configs[1..3] at their full sizes
def test_config2_lif_1000x1000_stdp(oracle_lattice_factory):
    """BASELINE.json configs[1]: leaky integrate-and-fire 1000 x 1000 with STDP (first steps; the oracle needs 0.1 s per step).
    The LIF step has no transcendental, so rasters and last_firing_time are exact; voltages and weights to STDP's expf rounding."""
    a, b = pair(oracle_lattice_factory, model="lif", rows=1000, cols=1000, seed=12, graph="grid", stdp=True, history=False, gap=40.0)
    b._be.set_option(K.OPT_PARALLEL, 1)   # parallel = true: the oracle gathers with OpenMP (80 ms per step)
    a.run_lattice(50)
    a.run_lattice(30)
    b.run_lattice(80)
    la, lb = a.get_field("last_firing_time"), b.get_field("last_firing_time")
    assert (lb >= 0).sum() > 10000 and (la == lb).all()
    assert (a.get_field("refractory_count") == b.get_field("refractory_count")).all()
    np.testing.assert_allclose(a.get_field("current_voltage"), b.get_field("current_voltage"), rtol=1e-5, atol=1e-4)
    (rpa, pa, wa), (rpb, pb, wb) = a.graph_csr(), b.graph_csr()
    assert (rpa == rpb).all() and (pa == pb).all() and wa.size == 8 * 10**6 - 6 * 2000 + 4
    np.testing.assert_allclose(wa, wb, rtol=1e-5, atol=1e-6)
    assert np.abs(wb - 1.0).max() > 1e-3


def test_config3_hodgkin_huxley_256x256_receptors(oracle_lattice_factory):
    """BASELINE.json configs[2]: Hodgkin-Huxley 256 x 256 with AMPA / NMDA / GABA receptors, Destexhe neurotransmitter and
    receptor kinetics, electrical + chemical synapses, dt = 0.01 (expf / powf everywhere: tolerance)."""
    a, b = pair(oracle_lattice_factory, model="hh", rows=256, cols=256, seed=13, graph="grid", chem="destexhe_all", history=False,
                gap=2.0)
    for L in (a, b):
        L.run_lattice(60)
    for name, tol in (("current_voltage", 1e-3), ("na_channel$m$state", 1e-5), ("na_channel$h$state", 1e-5), ("k_channel$n$state", 1e-5),
                      ("neurotransmitters$t", 1e-5), ("receptors$AMPA$r$kinetics$r", 1e-5), ("receptors$NMDA$r$kinetics$r", 1e-5),
                      ("receptors$GABA$r$kinetics$r", 1e-5), ("receptors$NMDA_current", 1e-3)):
        # the gate rates are singular at V = -40 / -55 mV (0/0 forms): an expf ulp is amplified for the handful of neurons that
        # sit next to the singularity, hence the robust form of allclose (at most 0.1 % of the cells, bounded in size)
        SC.assert_close_robust(a.get_field(name), b.get_field(name), 1e-4, tol, name, max_frac=0.001, max_abs=0.05)
    assert (a.get_field("was_increasing") == b.get_field("was_increasing")).all()
    assert (a.get_field("last_firing_time") == b.get_field("last_firing_time")).all()


def test_config4_mnist_shaped_network_full_size(oracle_lattice_factory, oracle_network_factory):
    """BASELINE.json configs[3] at its full size: 784 spike trains (28 x 28, all-to-all onto the excitatory lattice) -> 400
    excitatory <-> 400 inhibitory Izhikevich neurons, AMPA / GABA, STDP on both lattices.  Rate trains instead of Poisson so that
    the run is deterministic (Poisson parity is statistical, test_poisson_network_firing_statistics); wide-row kernel."""
    def build(lfac, nfac):
        rng = np.random.default_rng(1)
        T = S.IonotropicNeurotransmitterType
        exc_base = S.IzhikevichNeuron(gap_conductance=5.0, c_m=10.0)
        exc_base.synaptic_neurotransmitters[T.AMPA] = S.ApproximateNeurotransmitter()
        exc_base.receptors[T.AMPA] = S.AMPAReceptor()
        exc_base.receptors[T.GABA] = S.GABAReceptor()
        inh_base = exc_base.clone()
        inh_base.synaptic_neurotransmitters = {T.GABA: S.ApproximateNeurotransmitter()}
        exc = S.Lattice(S.IzhikevichNeuron, id=1, backend_factory=lfac)
        exc.populate(exc_base, 20, 20)
        inh = S.Lattice(S.IzhikevichNeuron, id=2, backend_factory=lfac)
        inh.populate(inh_base, 20, 20)
        for L in (exc, inh):
            L.set_field("current_voltage", rng.uniform(-65, 20, 400).astype(f32))
            L.set_field("b", rng.uniform(0.25, 0.33, 400).astype(f32))
            L.do_plasticity = True
            L.plasticity = S.STDP(a_plus=0.01, a_minus=0.01)
            L.update_grid_history = L.update_spike_history = True
        base = S.RateSpikeTrain(rate=2.0)
        base.synaptic_neurotransmitters[T.AMPA] = S.ApproximateNeurotransmitter()
        st = S.SpikeTrainLattice(S.RateSpikeTrain, id=0, network_backend_factory=nfac)
        st.populate(base, 28, 28)
        st.set_field("rate", rng.choice([0.0, 1.5, 2.0, 3.0, 5.0], 784).astype(f32))
        net = S.LatticeNetwork.generate_network([exc, inh], [st], backend_factory=nfac)
        w = rng.uniform(0, 1, (784, 400)).astype(f32)
        net.connect(0, 1, lambda x, y: True, lambda x, y: float(w[x[0] * 28 + x[1], y[0] * 20 + y[1]]))
        net.connect(1, 2, lambda x, y: x == y, lambda x, y: 1.0)
        net.connect(2, 1, lambda x, y: x != y, lambda x, y: -1.0)
        net.electrical_synapse, net.chemical_synapse = True, True
        return net
    a, b = build(None, None), build(oracle_lattice_factory, oracle_network_factory)
    a.run_lattices(40)
    b.run_lattices(40)
    spikes = 0
    for lid in (1, 2):
        ha, hb = a.get_lattice(lid).grid_history.history, b.get_lattice(lid).grid_history.history
        SC.assert_close_robust(ha, hb, 1e-4, 1e-3, f"lattice {lid}")
        ra, rb = a.get_lattice(lid).spike_history.history, b.get_lattice(lid).spike_history.history
        assert (ra == rb).all()
        spikes += int(rb.sum())
    assert spikes > 50
    for pre, post in ((0, 1), (1, 2), (2, 1)):
        (ca, wa), (cb, wb) = a._be.get_connection_dense(pre, post), b._be.get_connection_dense(pre, post)
        assert (ca == cb).all() and int(cb.sum()) == {(0, 1): 313600, (1, 2): 400, (2, 1): 159600}[(pre, post)]
        np.testing.assert_allclose(wa, wb, rtol=1e-5, atol=1e-6, err_msg=f"weights {pre}->{post}")


# ------------------------------------------------------------------ full size (BASELINE.json configs[4] shape)
def _window_check(big, rows, cols, r0, c0, h, w, k, oracle_lattice_factory, init, extra_fields=()):
    """The state of a neuron after k steps depends only on cells within Chebyshev distance k (radius-1 stencil), so a
    (h+2k)x(w+2k) patch stepped by the oracle must reproduce the big lattice's window exactly."""
    ra, rb = max(0, r0 - k), min(rows, r0 + h + k)
    ca, cb = max(0, c0 - k), min(cols, c0 + w + k)
    # a patch edge that is not a lattice edge gets wrong neighbours: keep only cells at distance >= k from such edges
    patch = SC.build_lattice(oracle_lattice_factory, model="izh", rows=rb - ra, cols=cb - ca, seed=0, graph="grid", hetero=False,
                             history=False)
    for name, arr in init.items():
        patch.set_field(name, arr.reshape(rows, cols)[ra:rb, ca:cb])
    patch.run_lattice(k)
    for name in ("current_voltage", "w_value", "last_firing_time") + tuple(extra_fields):
        got = big.get_field(name).reshape(rows, cols)[r0:r0 + h, c0:c0 + w]
        want = patch.get_field(name).reshape(rb - ra, cb - ca)[r0 - ra:r0 - ra + h, c0 - ca:c0 - ca + w]
        assert (got == want).all(), name


def test_full_size_10m_izhikevich_window_property(oracle_lattice_factory):
    """Electrical synapses only: no transcendental anywhere, every compared field bit for bit after k = 24 steps."""
    rows = cols = 3163
    n = rows * cols
    rng = np.random.default_rng(2024)
    init = {"current_voltage": rng.uniform(-65, 30, n).astype(f32), "b": rng.uniform(0.25, 0.36, n).astype(f32)}
    big = SC.build_lattice(None, model="izh", rows=rows, cols=cols, seed=0, graph="grid", hetero=False, history=False)
    big.fill_field("c_m", 2.0)
    for name, arr in init.items():
        big.set_field(name, arr)
    k = 24
    big.run_lattice(k)
    assert big.internal_clock == k
    init["c_m"] = np.full(n, 2.0, f32)
    for (r0, c0) in [(0, 0), (1500, 1700), (rows - 16, cols - 16), (0, cols - 16), (3000, 0)]:
        _window_check(big, rows, cols, r0, c0, 16, 16, k, oracle_lattice_factory, init)
    spikes = (big.get_field("last_firing_time") >= 0).sum()
    assert spikes > 1000


def _bench_config_lattice(factory, rows, cols, init):
    """The bench workload (bench.py, BASELINE.json configs[4] shape): Izhikevich, radius-1 Moore grid, electrical + AMPA chemistry
    (ApproximateNeurotransmitter / ApproximateReceptor), STDP on."""
    lat = SC.build_lattice(factory, model="izh", rows=rows, cols=cols, seed=0, graph="grid", hetero=False, history=False,
                           chem="approx_ampa", stdp=True, c_m=2.0)
    lat.plasticity = S.STDP(a_plus=0.05, a_minus=0.04, tau_plus=4.5, tau_minus=3.0)
    for name, arr in init.items():
        lat.set_field(name, arr)
    return lat


BENCH_STATE = ("current_voltage", "w_value", "last_firing_time", "neurotransmitters$t", "receptors$AMPA$r$kinetics$r")


def _bench_window_check(big, rows, cols, r0, c0, h, w, k, factory, init):
    """Light cone: after k steps a cell depends only on cells within Chebyshev distance k, so a (h+2k) x (w+2k) patch stepped by
    the oracle must reproduce the window — last_firing_time bit for bit, float state to 1e-4 (STDP's expf is the one
    transcendental), weights of the window's in-edges to 1e-4."""
    ra, rb = max(0, r0 - k), min(rows, r0 + h + k)
    ca, cb = max(0, c0 - k), min(cols, c0 + w + k)
    patch = _bench_config_lattice(factory, rb - ra, cb - ca, {n_: a.reshape(rows, cols)[ra:rb, ca:cb] for n_, a in init.items()})
    patch.run_lattice(k)
    pc = cb - ca
    for name in BENCH_STATE:
        got = big[name].reshape(rows, cols, -1)[r0:r0 + h, c0:c0 + w]
        want = patch.get_field(name).reshape(rb - ra, pc, -1)[r0 - ra:r0 - ra + h, c0 - ca:c0 - ca + w]
        if name == "last_firing_time":
            assert (got == want).all(), (name, r0, c0)
        else:
            np.testing.assert_allclose(got, want, rtol=1e-4, atol=1e-4, err_msg=f"{name} at ({r0},{c0})")
    prp, ppre, pw = patch._be.get_connection_csr()
    changed = 0
    for r in range(r0, r0 + h):
        rp, pre, ww = big["rows"](r * cols + c0, r * cols + c0 + w)
        for q in range(w):
            pq = (r - ra) * pc + (c0 + q - ca)
            s, t = int(prp[pq]), int(prp[pq + 1])
            gpre = pre[int(rp[q]):int(rp[q + 1])]
            # same in-edges (global index -> patch index) and the same weights
            assert ((gpre // cols - ra) * pc + (gpre % cols - ca) == ppre[s:t]).all()
            np.testing.assert_allclose(ww[int(rp[q]):int(rp[q + 1])], pw[s:t], rtol=1e-4, atol=1e-5)
            changed += int((np.abs(pw[s:t] - 1.0) > 1e-6).sum())
    return changed


def _full_size_bench_config(rows, cols, k, windows, factory, seed):
    n = rows * cols
    rng = np.random.default_rng(seed)
    init = {"current_voltage": rng.uniform(-65, 30, n).astype(f32), "b": rng.uniform(0.25, 0.36, n).astype(f32)}
    lat = _bench_config_lattice(None, rows, cols, init)
    lat.run_lattice(k)
    assert lat.internal_clock == k
    big = {name: lat.get_field(name) for name in BENCH_STATE}
    big["rows"] = lat._be.get_graph_rows
    changed = 0
    for (r0, c0) in windows:
        changed += _bench_window_check(big, rows, cols, r0, c0, 16, 16, k, factory, init)
    assert (big["last_firing_time"] >= 0).sum() > 1000
    assert changed > 0, "STDP never changed a weight inside the windows"
    assert np.abs(big["neurotransmitters$t"]).max() > 0


def test_full_size_10m_bench_config_window_property(oracle_lattice_factory):
    """BASELINE.json configs[4] shape as bench.py runs it (3163 x 3163 Izhikevich, electrical + AMPA + STDP) through the
    window-staged kernel at full size: five 16 x 16 windows incl. corners and edges, k = 12 steps."""
    rows = cols = 3163
    _full_size_bench_config(rows, cols, 12, [(0, 0), (1500, 1700), (rows - 16, cols - 16), (0, cols - 16), (3000, 0)],
                            oracle_lattice_factory, 2024)


def test_full_size_100m_bench_config_window_property(oracle_lattice_factory):
    """The same property at 10^8 neurons on one GPU (10 000 x 10 000, ~25 GB of HBM): 64-bit offsets, node indices near the
    28-bit limit of the col words."""
    rows = cols = 10000
    _full_size_bench_config(rows, cols, 6, [(0, 0), (rows // 2 + 3, cols // 2 - 5), (rows - 16, cols - 16)], oracle_lattice_factory, 5)


def test_full_size_uniform_state_follows_isolated_neuron(oracle_lattice_factory):
    """Identical neurons => zero gap current => every one of the 10^7 neurons follows the isolated trajectory
    (the size-independent form of tests/gpu_connection_behavior.rs:51-95)."""
    rows = cols = 3163
    big = SC.build_lattice(None, model="izh", rows=rows, cols=cols, seed=0, graph="grid", hetero=False, history=False)
    iso = SC.build_lattice(oracle_lattice_factory, model="izh", rows=1, cols=1, seed=0, graph="none", hetero=False, history=False)
    for L in (big, iso):
        L.fill_field("current_voltage", -40.0)
        L.fill_field("b", 0.35)
        L.fill_field("c_m", 1.0)
        L.fill_field("w_value", -5.0)
    big.run_lattice(400)
    iso.run_lattice(400)
    v = big.get_field("current_voltage")
    assert (v == iso.get_field("current_voltage")[0]).all()
    assert (big.get_field("last_firing_time") == iso.get_field("last_firing_time")[0]).all()
    assert iso.get_field("last_firing_time")[0] >= 0
