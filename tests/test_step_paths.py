"""Whole-lattice oracle parity of every step path at the sizes that select it.

A timestep is computed by one of five step paths (Engine::plan_step_path): the window-staged and the TMA-staged persistent
kernels for stencil lattices of at least 64 Ki neurons, the one-CTA-per-slice wide kernel and its two-pass split for wide rows,
and the one-thread-per-neuron general kernel; General and Wide also run whole chunks of timesteps in one cooperative launch
(step_multi.cu), in a 16-CTA cluster (at most 320 slices), on a grid barrier with one slice per warp, or grid-striding with
several slices per warp.  The loops that only run at scale (stage rings that wrap, many tiles per CTA, the reversed tile order
of odd steps, the grid barrier, grid-stride loops, the sum-pass ring of very wide rows) are compared here, every cell, with
the CPU oracle.  Each case asserts the path it ran (SNN_OPT_STEP_PATH), so that a threshold change cannot move a case to
another path unnoticed.
"""
import numpy as np
import pytest

import scenarios as SC
import snn_b200 as S
from snn_b200 import _capi as K

pytestmark = pytest.mark.gpu
f32 = np.float32

GEN, WIDE, SPLIT, TMA, WIN, MULTI = (K.STEP_PATH_GENERAL, K.STEP_PATH_WIDE, K.STEP_PATH_WIDE_SPLIT, K.STEP_PATH_TMA,
                                     K.STEP_PATH_WIN, K.STEP_PATH_MULTI)


@pytest.fixture
def kernel_env(monkeypatch):
    """Sets SNN_B200_TMA / SNN_B200_WIN for one case (None: the automatic choice)."""
    def set_env(tma=None, win=None):
        for name, v in (("SNN_B200_TMA", tma), ("SNN_B200_WIN", win)):
            if v is None:
                monkeypatch.delenv(name, raising=False)
            else:
                monkeypatch.setenv(name, str(v))
    set_env()
    return set_env


def local_csr(rows, cols, radius, p, hubs=(), hub_in=0, empty=(), *, seed):
    """Random local graph in CSR (rows = postsynaptic neurons, presynaptic indices ascending): an edge from every neuron within
    Euclidean distance `radius` with probability p, plus `hub_in` random in-edges for each neuron of `hubs`, minus every
    in-edge of the neurons of `empty`.  Weights are drawn in [0.2, 2] and divided by a tenth of the row's in-degree, so that
    wide rows drive their neuron about as hard as the 8-neighbour grid does."""
    rng = np.random.default_rng(seed)
    n = rows * cols
    r, c = np.divmod(np.arange(n, dtype=np.int64), cols)
    ri = int(np.floor(radius))
    posts, pres = [], []
    for dr in range(-ri, ri + 1):
        for dc in range(-ri, ri + 1):
            if (dr, dc) == (0, 0) or np.hypot(dr, dc) > radius:
                continue
            pr, pc = r + dr, c + dc
            ok = (pr >= 0) & (pr < rows) & (pc >= 0) & (pc < cols) & (rng.random(n) <= p)
            posts.append(np.nonzero(ok)[0])
            pres.append((pr * cols + pc)[ok])
    for h in hubs:
        src = rng.choice(n, hub_in + 1, replace=False)
        src = src[src != h][:hub_in]
        posts.append(np.full(src.size, h, np.int64))
        pres.append(src)
    key = np.unique(np.concatenate(posts) * n + np.concatenate(pres))
    post, pre = np.divmod(key, n)
    keep = ~np.isin(post, np.asarray(empty, np.int64))
    post, pre = post[keep], pre[keep]
    deg = np.bincount(post, minlength=n)
    row_ptr = np.zeros(n + 1, np.uint64)
    row_ptr[1:] = np.cumsum(deg)
    w = (rng.uniform(0.2, 2.0, post.size) / np.maximum(deg[post] / 10.0, 1.0)).astype(f32)
    return row_ptr, pre.astype(np.uint32), w


# ------------------------------------------------------------------ specialisations
# (model, chemistry, plasticity): plasticity None, "stdp" or "bcm"
ELECTRICAL = [(m, None, None) for m in SC.MODELS]
WIN_SPECS = ELECTRICAL + [("izh", "approx_ampa", None), ("izh", "approx_all", "stdp"), ("lif", "expdecay_all", None),
                          ("qif", "discrete_ampa", None), ("hh", "destexhe_all", None), ("lif", None, "stdp"),
                          ("bcm_izh", None, "bcm")]
MULTI_GRID_SPECS = [("izh", None, None), ("izh", None, "stdp"), ("izh", "approx_all", None), ("hh", "destexhe_all", None)]
MULTI_SLICES_SPECS = [("izh", None, None), ("izh", None, "stdp"), ("lif", "approx_ampa", None), ("hh", None, None)]
WIDE_SPECS = [("izh", None, None), ("izh", "approx_ampa", None), ("izh", "approx_all", "stdp"), ("hh", "destexhe_all", None),
              ("bcm_izh", None, "bcm")]


def spec_id(spec):
    return "-".join(x for x in spec if x)


def is_exact(spec):
    """Models and chemistry without a transcendental and without STDP (whose weight update calls expf): bit for bit."""
    model, chem, plast = spec
    return model in SC.EXACT_MODELS and chem in (None, "approx_ampa") and plast != "stdp"


def win_rows(spec):
    """Rows of a cols = 1000 lattice for the window kernel: ~1 M neurons give each CTA ~28 tiles, enough for the 8-stage ring of
    the small-stage specialisations to wrap three times; the large stages of Hodgkin-Huxley and of chemistry give few stages,
    for which 262 rows (~2 tiles per CTA and stage) wrap the ring as well."""
    model, chem, _ = spec
    return 262 if model == "hh" or chem else 1024


def build(factory, spec, rows, cols, graph, seed):
    model, chem, plast = spec
    if isinstance(graph, tuple):   # local_csr arguments
        lat = SC.build_lattice(factory, model=model, rows=rows, cols=cols, seed=seed, graph="none", chem=chem,
                               stdp=plast is not None, gap=SC.drive_current(model))
        lat.connect_csr(*local_csr(rows, cols, *graph, seed=seed + 100))
    else:
        lat = SC.build_lattice(factory, model=model, rows=rows, cols=cols, seed=seed, graph=graph, chem=chem,
                               stdp=plast is not None, gap=SC.drive_current(model))
    if plast == "stdp":
        lat.plasticity = S.STDP(a_plus=0.05, a_minus=0.04, tau_plus=4.5, tau_minus=3.0, dt=0.1)
    elif plast == "bcm":
        # dt = 1e-4: the weights move by more than their rounding within a few dozen steps
        lat.plasticity = S.BCM(decay=0.05, average_scalar=0.5, dt=1e-4)
    return lat


def segments_of(spec, short):
    """Run calls of odd and even length (the ping-pong parities continue across calls).  Exact specs run the whole horizon in
    two calls.  The others are chaotic: an ulp of expf grows to millivolts within a few hundred steps (the oracle and the
    numpy restatement diverge the same way), so they run in segments of 25 / 24 steps, each compared to the config-3 bars
    and followed by a re-synchronisation of the device from the oracle (the pattern of scenarios.lockstep_lattices).
    Hodgkin-Huxley runs 61 steps (dt = 0.01), as config 3 does: whole lattices of it reach the reference's singular gate
    rates (non-finite voltages) within tens to hundreds of steps, before their first action potentials (~420 steps)."""
    total = 61 if spec[0] == "hh" else (25 if short else 301)
    if is_exact(spec):
        return [total // 2 + 1, total - total // 2 - 1]
    seg = (13, 12) if total == 25 else ((31, 30) if total == 61 else (25, 24))
    out = []
    while sum(out) < total:
        out.append(min(seg[len(out) % 2], total - sum(out)))
    return out


def compare(a, b, spec, lo, hi):
    """a = device, b = oracle: every cell of the grid history of steps [lo, hi), the raster, every state field and the
    weights."""
    exact = is_exact(spec)
    ha, hb = a.grid_history.history[lo:hi], b.grid_history.history[lo:hi]
    assert ha.shape == hb.shape and ha.shape[0] == hi - lo
    sa, sb = a.spike_history.history[lo:hi], b.spike_history.history[lo:hi]
    if exact:
        bad = np.nonzero(ha != hb)
        assert bad[0].size == 0, f"{bad[0].size} voltages differ, first at step {lo + bad[0][0]} cell ({bad[1][0]},{bad[2][0]})"
        assert (sa == sb).all(), f"raster differs at steps {lo + np.unique(np.nonzero(sa != sb)[0])[:5]}"
    else:
        SC.assert_close_robust(ha, hb, 1e-4, 1e-3, f"grid history of steps {lo}..{hi}", max_frac=0.001, max_abs=0.05)
        if spec[0] in SC.EXACT_MODELS:   # STDP on an exact model: the threshold crossings still agree
            assert (sa == sb).all(), f"raster differs at steps {lo + np.unique(np.nonzero(sa != sb)[0])[:5]}"
    assert (a.get_field("last_firing_time") == b.get_field("last_firing_time")).all(), f"last_firing_time after step {hi}"
    for name in SC.lattice_field_names(b):
        fa, fb = a.get_field(name), b.get_field(name)
        assert fa.shape == fb.shape, name
        if exact or fa.dtype.kind in "iu":
            assert (fa == fb).all(), f"{name} after step {hi}: {(fa != fb).sum()} of {fa.size} cells differ"
        else:
            tol = 1e-3 if ("voltage" in name or "current" in name) else 1e-5
            SC.assert_close_robust(fa, fb, 1e-4, tol, f"{name} after step {hi}", max_frac=0.001, max_abs=0.05)
    (rpa, pa, wa), (rpb, pb, wb) = a.graph_csr(), b.graph_csr()
    assert (rpa == rpb).all() and (pa == pb).all()
    if spec[2] == "stdp":
        np.testing.assert_allclose(wa, wb, rtol=1e-5, atol=1e-6, err_msg=f"weights after step {hi}")
    else:
        assert (wa == wb).all(), f"weights after step {hi}"


def run_parity(oracle_lattice_factory, spec, rows, cols, graph, expect, seed=5, short=True, spg=None):
    a = build(None, spec, rows, cols, graph, seed)
    b = build(oracle_lattice_factory, spec, rows, cols, graph, seed)
    b._be.set_option(K.OPT_PARALLEL, 1)
    if spg is not None:
        a._be.set_option(K.OPT_STEPS_PER_GRAPH, spg)
    w0 = b.graph_csr()[2].copy()
    assert a._be.get_option(K.OPT_STEP_PATH) == K.STEP_PATH_NONE
    paths, done = [], 0
    for k in segments_of(spec, short):
        a.run_lattice(k)
        b.run_lattice(k)
        paths.append(a._be.get_option(K.OPT_STEP_PATH))
        compare(a, b, spec, done, done + k)
        done += k
        if not is_exact(spec):   # the weights stay: they differ by roundings, which the state no longer amplifies
            SC.copy_lattice_state(b, a, weights=False)
    if spec[0] == "hh":   # no action potential yet (segments_of): the subthreshold dynamics must be under way
        h = b.grid_history.history
        assert np.nanmax(np.abs(h - h[0])) > 0.1, "the scenario must move the voltages"
    else:
        assert b.spike_history.history.sum() > 0, "the scenario must spike"
    if spec[2] is not None:   # 1e-6: several roundings of the largest weights (2.0)
        assert np.abs(b.graph_csr()[2] - w0).max() > 1e-6, "plasticity must move weights"
    assert paths == [expect] * len(paths), f"step path {paths}, expected {expect}"


# ------------------------------------------------------------------ persistent kernels, rings that wrap
@pytest.mark.parametrize("spec", WIN_SPECS, ids=spec_id)
def test_window_kernel_ring_wraps(spec, kernel_env, oracle_lattice_factory):
    run_parity(oracle_lattice_factory, spec, win_rows(spec), 1000, "grid", WIN)


@pytest.mark.parametrize("cols", [255, 256, 257, 258, 259, 1021])
def test_window_kernel_geometry(cols, kernel_env, oracle_lattice_factory):
    """Row lengths around the 256-neuron tile and every residue mod 4: the window rows of a tile straddle lattice rows."""
    rows = -(-65536 // cols) + 1
    run_parity(oracle_lattice_factory, ("izh", None, "stdp"), rows, cols, "grid", WIN, seed=cols)


@pytest.mark.parametrize("spec", WIN_SPECS, ids=spec_id)
@pytest.mark.parametrize("how", ["radius2", "radius1_win0"])
def test_tma_kernel_ring_wraps(how, spec, kernel_env, oracle_lattice_factory):
    """~590 K neurons: ~5 tiles per CTA for three CTAs per SM and up to four stages."""
    if how == "radius1_win0":
        kernel_env(win=0)
    rows = 262 if spec[0] == "hh" or spec[1] else 590
    run_parity(oracle_lattice_factory, spec, rows, 1000, "grid2" if how == "radius2" else "grid", TMA)


# ------------------------------------------------------------------ cooperative multi-step kernel beyond one cluster
@pytest.mark.parametrize("spec", MULTI_GRID_SPECS, ids=spec_id)
def test_multi_grid_barrier_one_slice_per_warp(spec, kernel_env, oracle_lattice_factory):
    """150 x 151 = 22 650 neurons, 708 slices: more than one cluster holds, fewer than one warp each needs the grid to stride;
    the whole run is one cooperative launch on the grid barrier.  Izhikevich without plasticity takes the register-cached rows."""
    run_parity(oracle_lattice_factory, spec, 150, 151, "grid", GEN + MULTI, short=False, spg=0)


LARGE_GRAPHS = {"csr": (2.0, 0.8), "grid": "grid"}


def large_expect(spec, spg):
    return GEN if spg == 1 else GEN + MULTI


@pytest.mark.parametrize("spec", MULTI_SLICES_SPECS, ids=spec_id)
@pytest.mark.parametrize("graph", list(LARGE_GRAPHS))
@pytest.mark.parametrize("spg", [0, 1])
def test_general_large(spg, graph, spec, kernel_env, oracle_lattice_factory):
    """400 x 640 = 256 000 neurons, 8 000 slices: with spg 0 the multi-step kernel grid-strides with several slices per warp
    (the grid-stride loop, and for Izhikevich without plasticity the register-cached rows past the first pass); with spg 1 the
    general kernel runs one launch per step at scale.  The radius-1 grid is kept off the staged kernels with SNN_B200_TMA=0.
    The size keeps every spec in the multi-step regime on 148 SMs: more than 8 and at most 32 slices per resident CTA (8 warps
    each) for three resident CTAs per SM (Izhikevich, 80 registers) as for two (the others, 100 to 124 registers)."""
    kernel_env(tma=0)
    run_parity(oracle_lattice_factory, spec, 400, 640, LARGE_GRAPHS[graph], large_expect(spec, spg), spg=spg)


# ------------------------------------------------------------------ wide rows
def wide_expect(spec, spg):
    # BCM runs its per-edge pass after every step: never the multi-step launch
    return WIDE if spg == 1 or spec[2] == "bcm" else WIDE + MULTI


@pytest.mark.parametrize("spec", WIDE_SPECS, ids=spec_id)
@pytest.mark.parametrize("shape", [(64, 64), (120, 120)], ids=["staged", "global"])
@pytest.mark.parametrize("spg", [0, 1])
def test_wide(spg, shape, spec, kernel_env, oracle_lattice_factory):
    """Radius 5, p = 0.9: ~70 in-edges per neuron (mean slice width between 48 and 119 k-rows).  4 096 neurons stage the node
    state in shared memory; 14 400 (450 slices) read it from global memory, and the multi-step kernel grid-strides past its
    resident CTAs (one to three per SM of 512 threads, depending on the registers and the chunk buffers of the spec)."""
    run_parity(oracle_lattice_factory, spec, *shape, (5.0, 0.9), wide_expect(spec, spg), spg=spg)


@pytest.mark.parametrize("spec", WIDE_SPECS, ids=spec_id)
def test_wide_split(spec, kernel_env, oracle_lattice_factory):
    """Radius 8, p = 0.9 (~180 in-edges): the two-pass kernel.  Hub rows of 600 in-edges wrap the sum pass's ring of
    kWideSumBufs 60-row chunk buffers; next to them rows without any in-edge."""
    rows, cols = 140, 143
    hubs = [0, 1, 777, 5000, rows * cols - 1]
    empty = [2, 3, 778, 5001, 5002, rows * cols - 2]
    run_parity(oracle_lattice_factory, spec, rows, cols, (8.0, 0.9, hubs, 600, empty), SPLIT)


# ------------------------------------------------------------------ network on the grid barrier
def build_big_network(lattice_factory, network_factory, side=120, st_side=16, seed=31):
    """The shape of test_gpu_parity.build_network at 2 x 120 x 120 neurons: rate trains -> excitatory <-> inhibitory, AMPA /
    GABA, STDP on both lattices.  Sparse local connections in CSR (the dense connect of the small network is n^2)."""
    rng = np.random.default_rng(seed)
    T = S.IonotropicNeurotransmitterType
    n = side * side
    exc_base = S.IzhikevichNeuron(gap_conductance=5.0, c_m=10.0)
    exc_base.synaptic_neurotransmitters[T.AMPA] = S.ApproximateNeurotransmitter()
    exc_base.receptors[T.AMPA] = S.AMPAReceptor()
    exc_base.receptors[T.GABA] = S.GABAReceptor()
    inh_base = exc_base.clone()
    inh_base.synaptic_neurotransmitters = {T.GABA: S.ApproximateNeurotransmitter(clearance_constant=0.02)}
    exc = S.Lattice(S.IzhikevichNeuron, id=1, backend_factory=lattice_factory)
    exc.populate(exc_base, side, side)
    inh = S.Lattice(S.IzhikevichNeuron, id=2, backend_factory=lattice_factory)
    inh.populate(inh_base, side, side)
    for L in (exc, inh):
        L.set_field("current_voltage", rng.uniform(-65, 20, n).astype(f32))
        L.set_field("b", rng.uniform(0.25, 0.33, n).astype(f32))
        L.update_grid_history = L.update_spike_history = True
        L.do_plasticity = True
        L.plasticity = S.STDP(a_plus=0.03, a_minus=0.03)
    base = S.RateSpikeTrain(rate=2.0)
    base.synaptic_neurotransmitters[T.AMPA] = S.ApproximateNeurotransmitter()
    st = S.SpikeTrainLattice(S.RateSpikeTrain, id=0, network_backend_factory=network_factory)
    n_st = st_side * st_side
    st.populate(base, st_side, st_side)
    st.set_field("rate", rng.choice([0.0, 1.5, 2.0, 3.0], n_st).astype(f32))
    st.update_spike_history = True
    net = S.LatticeNetwork.generate_network([exc, inh], [st], backend_factory=network_factory)
    be = net._be
    be.connect_csr(1, 1, *local_csr(side, side, 1.0, 1.0, seed=seed + 1))
    # every excitatory neuron hears 8 random trains
    pre = np.sort(np.stack([rng.choice(n_st, 8, replace=False) for _ in range(n)]), axis=1).astype(np.uint32).ravel()
    be.connect_csr(0, 1, np.arange(0, 8 * n + 1, 8, dtype=np.uint64), pre, rng.uniform(0, 1, 8 * n).astype(f32))
    be.connect_csr(1, 2, np.arange(n + 1, dtype=np.uint64), np.arange(n, dtype=np.uint32), np.ones(n, f32))
    rp, pr, _ = local_csr(side, side, 2.0, 0.5, seed=seed + 2)
    be.connect_csr(2, 1, rp, pr, np.full(pr.size, -1.0, f32))
    net.electrical_synapse, net.chemical_synapse = True, True
    return net


NET_PAIRS = ((0, 1), (1, 1), (1, 2), (2, 1))


def test_network_grid_barrier(kernel_env, oracle_lattice_factory, oracle_network_factory):
    """28 800 neurons and 256 trains in one cooperative launch per run call on the grid barrier; STDP with spike trains makes
    the kernel wait for every neuron before the trains step (train_sync)."""
    a = build_big_network(None, None)
    b = build_big_network(oracle_lattice_factory, oracle_network_factory)
    b._be.set_option(K.OPT_PARALLEL, 1)
    a._be.set_option(K.OPT_STEPS_PER_GRAPH, 0)
    w0 = {pp: b._be.get_connection_csr(*pp)[2].copy() for pp in NET_PAIRS}
    paths = []
    for k in (41, 40):
        a.run_lattices(k)
        b.run_lattices(k)
        paths.append(a._be.get_option(K.OPT_STEP_PATH))
    sa, sb = a.get_spike_train_lattice(0).spike_history.history, b.get_spike_train_lattice(0).spike_history.history
    assert (sa == sb).all()
    spikes = 0
    for lid in (1, 2):
        la, lb = a.get_lattice(lid), b.get_lattice(lid)
        SC.assert_close_robust(la.grid_history.history, lb.grid_history.history, 1e-4, 1e-3, f"lattice {lid}", max_frac=0.001,
                               max_abs=0.05)
        assert (la.spike_history.history == lb.spike_history.history).all(), f"lattice {lid}: raster"
        assert (la.get_field("last_firing_time") == lb.get_field("last_firing_time")).all()
        spikes += int(lb.spike_history.history.sum())
    assert spikes > 100
    for pp in NET_PAIRS:
        (rpa, pa, wa), (rpb, pb, wb) = a._be.get_connection_csr(*pp), b._be.get_connection_csr(*pp)
        assert (rpa == rpb).all() and (pa == pb).all()
        np.testing.assert_allclose(wa, wb, rtol=1e-5, atol=1e-6, err_msg=f"weights {pp}")
    assert np.abs(b._be.get_connection_csr(0, 1)[2] - w0[(0, 1)]).max() > 1e-4
    assert paths == [GEN + MULTI] * 2


# ------------------------------------------------------------------ the path table in one place
def _small_network():
    from test_gpu_parity import build_network
    return build_network(None, None, st_shape=(16, 16))


def _path_table():
    """(name, environment, builder of the device handle, steps per graph, expected SNN_OPT_STEP_PATH)."""
    rows = []
    for spec in WIN_SPECS:
        rows.append((f"win-{spec_id(spec)}", {}, lambda s=spec: build(None, s, win_rows(s), 1000, "grid", 5), None, WIN))
        rows.append((f"tma-r2-{spec_id(spec)}", {}, lambda s=spec: build(None, s, 262, 1000, "grid2", 5), None, TMA))
        rows.append((f"tma-win0-{spec_id(spec)}", {"win": 0}, lambda s=spec: build(None, s, 262, 1000, "grid", 5), None, TMA))
    rows.append(("win-geometry-257", {}, lambda: build(None, ("izh", None, "stdp"), 256, 257, "grid", 5), None, WIN))
    for spec in MULTI_GRID_SPECS:
        rows.append((f"multi-grid-{spec_id(spec)}", {}, lambda s=spec: build(None, s, 150, 151, "grid", 5), 0, GEN + MULTI))
    for spec in MULTI_SLICES_SPECS:
        for g in LARGE_GRAPHS:
            for spg in (0, 1):
                rows.append((f"large-{g}-spg{spg}-{spec_id(spec)}", {"tma": 0},
                             lambda s=spec, g=g: build(None, s, 400, 640, LARGE_GRAPHS[g], 5), spg, large_expect(spec, spg)))
    for spec in WIDE_SPECS:
        for shape in ((64, 64), (120, 120)):
            for spg in (0, 1):
                rows.append((f"wide-{shape[0]}-spg{spg}-{spec_id(spec)}", {},
                             lambda s=spec, sh=shape: build(None, s, *sh, (5.0, 0.9), 5), spg, wide_expect(spec, spg)))
        rows.append((f"wide-split-{spec_id(spec)}", {},
                     lambda s=spec: build(None, s, 140, 143, (8.0, 0.9, [0, 777], 600, [2, 778]), 5), None, SPLIT))
    rows.append(("network-120x120", {}, lambda: build_big_network(None, None), 0, GEN + MULTI))
    # the small suite scenarios: a 7 x 9 grid is stepped by the 16-CTA cluster variant of the multi-step kernel, the
    # all-to-all 7 x 9 lattice (62 in-edges) by the multi-step wide kernel, the 256-train network's wide rows by the split kernel
    rows.append(("suite-7x9-grid", {}, lambda: SC.build_lattice(None, model="izh", rows=7, cols=9, graph="grid"), None, GEN + MULTI))
    rows.append(("suite-7x9-all", {}, lambda: SC.build_lattice(None, model="izh", rows=7, cols=9, graph="all"), None, WIDE + MULTI))
    rows.append(("suite-network-16x16-trains", {}, _small_network, None, SPLIT))
    return rows


def test_path_table(kernel_env):
    """One step of every scenario above and of three small suite scenarios; every recorded path at once in the message."""
    got, want = {}, {}
    for name, env, make, spg, expect in _path_table():
        kernel_env(**env)
        h = make()
        if spg is not None:
            h._be.set_option(K.OPT_STEPS_PER_GRAPH, spg)
        assert h._be.get_option(K.OPT_STEP_PATH) == K.STEP_PATH_NONE
        (h.run_lattices if hasattr(h, "run_lattices") else h.run_lattice)(1)
        got[name], want[name] = h._be.get_option(K.OPT_STEP_PATH), expect
        del h
    wrong = {k: (got[k], want[k]) for k in got if got[k] != want[k]}
    assert not wrong, f"(recorded, expected) step paths: {wrong}; all recorded: {got}"


def test_step_path_is_read_only():
    lat = SC.build_lattice(None, model="izh", rows=4, cols=4, graph="grid")
    with pytest.raises(K.SnnError) as e:
        lat._be.set_option(K.OPT_STEP_PATH, 1)
    assert e.value.status == K.SNN_INVALID_ARGUMENT
