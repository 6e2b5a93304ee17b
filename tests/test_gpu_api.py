"""Boundary behaviour of the C ABI on the device: SoA conversion round trips, graph ingestion, error codes, empty
lattices.  Mirrors the reference's conversion / edge-case tests (backend/tests/{neuron,neurotransmitter,ligand_gates,
spike_train}_conversion.rs, size_zero_cases.rs, grid_formation_invariant.rs)."""
import ctypes as C
import json
import os

import numpy as np
import pytest

import scenarios as SC
import snn_b200 as S
from snn_b200 import _capi as K
from snn_b200.backend import CudaLatticeBackend, CudaNetworkBackend

pytestmark = pytest.mark.gpu
f32 = np.float32
_NP = {K.F32: np.float32, K.U32: np.uint32, K.I32: np.int32}


def _random_for(name, dt, count, rng):
    if dt == K.F32:
        return rng.uniform(-3, 3, count).astype(f32)
    if dt == K.U32:
        return rng.integers(0, 2, count).astype(np.uint32)
    return rng.integers(-1, 1000, count).astype(np.int32)


@pytest.mark.parametrize("model", range(8))
@pytest.mark.parametrize("kin", [(0, 0), (1, 1), (3, 2), (2, 0)])
def test_every_field_round_trips(model, kin):
    """neuron_conversion.rs / neurotransmitter_conversion.rs / ligand_gates_conversion.rs: to-device then back equals
    the original, for every named field, including lattices that are not a multiple of the warp size."""
    be = CudaLatticeBackend(model, kin[0], kin[1], 5, 7)
    rng = np.random.default_rng(model * 10 + kin[0])
    vals = {}
    fields = be.fields(0)
    assert {"current_voltage", "gap_conductance", "dt", "is_spiking", "last_firing_time"} <= {f[0] for f in fields}
    for name, dt, per in fields:
        vals[name] = _random_for(name, dt, 35 * per, rng)
        be.set_field(0, name, vals[name])
    for name, dt, per in fields:
        got = be.get_field(0, name)
        assert got.dtype == _NP[dt] and (got == vals[name]).all(), name


def test_defaults_match_reference_default_impl(oracle_lattice_factory):
    """populate() with default_impl(): every field equals the Rust Default (and the oracle's independent table)."""
    for name, cls in SC.MODELS.items():
        be = CudaLatticeBackend(cls.model, cls.default_nt.kind, cls.default_rc.kind, 2, 3)
        ob = oracle_lattice_factory(cls.model, cls.default_nt.kind, cls.default_rc.kind, 2, 3)
        proto = cls()
        for fname, v in proto.scalar_fields().items():
            got = be.get_field(0, fname)
            want = -1 if v is None else v
            assert np.allclose(got, f32(want)), (name, fname)
            assert (got == ob.get_field(0, fname)).all(), (name, fname)
        for fname in ("receptors$AMPA_g", "receptors$NMDA_g", "receptors$NMDA_mg", "receptors$GABA_e", "neurotransmitters$t_max"):
            assert (be.get_field(0, fname) == ob.get_field(0, fname)).all(), (name, fname)


def test_field_errors():
    be = CudaLatticeBackend(K.MODEL_IZH, 0, 0, 3, 3)
    lib = be.lib
    a = np.zeros(9, f32)
    p = a.ctypes.data
    assert lib.snn_lattice_set_field(be.h, b"nonsense", p, 9, K.F32) == K.SNN_UNKNOWN_FIELD
    assert lib.snn_lattice_set_field(be.h, b"refractory_count", p, 9, K.F32) == K.SNN_UNKNOWN_FIELD  # not an Izhikevich field
    assert lib.snn_lattice_set_field(be.h, b"current_voltage", p, 8, K.F32) == K.SNN_SIZE_MISMATCH
    assert lib.snn_lattice_set_field(be.h, b"current_voltage", p, 9, K.U32) == K.SNN_DTYPE_MISMATCH
    assert lib.snn_lattice_set_field(be.h, b"neurotransmitters$t", p, 9, K.F32) == K.SNN_SIZE_MISMATCH
    assert b"current_voltage" in lib.snn_lattice_last_error(be.h) or b"neurotransmitters" in lib.snn_lattice_last_error(be.h)
    assert lib.snn_lattice_set_option(be.h, 1234, 1) == K.SNN_INVALID_ARGUMENT


def test_field_directory_order():
    """field_info(i) is public by index: the directory of every model x (neurotransmitter, receptor) kinetics lattice and of a
    network's spike-train lattice of every train kind x neurotransmitter kinetics is the one in golden/field_directory.json
    (`fields` holds the distinct (name, dtype, per) entries, each directory lists indices into it); index `count` is refused."""
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "field_directory.json")) as f:
        golden = json.load(f)
    entries = [tuple(e) for e in golden["fields"]]
    name, dt, per = C.c_char_p(), C.c_int32(), C.c_uint32()
    for key, want in golden["lattice"].items():
        model, ntk, rck = map(int, key.split())
        be = CudaLatticeBackend(model, ntk, rck, 2, 3)
        assert be.fields(0) == [entries[i] for i in want], key
        assert be.lib.snn_lattice_field_info(be.h, len(want), C.byref(name), C.byref(dt), C.byref(per)) == K.SNN_INVALID_ARGUMENT
        be.close()
    for key, want in golden["train"].items():
        kind, ntk = map(int, key.split())
        be = CudaNetworkBackend(K.MODEL_IZH, ntk, K.RC_APPROXIMATE, kind)
        be.add_train_lattice(7, 2, 3)
        assert be.fields(7) == [entries[i] for i in want], key
        assert be.lib.snn_network_field_info(be.h, 7, len(want), C.byref(name), C.byref(dt), C.byref(per)) == K.SNN_INVALID_ARGUMENT
        be.close()


def test_graph_ingestion_round_trips():
    rows, cols = 4, 5
    n = rows * cols
    conn, w = SC.random_graph(rows, cols, 5, weights="rand")
    be = CudaLatticeBackend(K.MODEL_IZH, 0, 0, rows, cols)
    be.connect_dense(0, 0, conn, w)
    c2, w2 = be.get_connection_dense()
    assert (c2 == conn).all() and (w2 == w).all()
    rp, pre, ww = SC.dense_to_csr(conn, w)
    # shuffled rows must come back canonical (presynaptic ascending)
    rng = np.random.default_rng(0)
    pre_s, ww_s = pre.copy(), ww.copy()
    for q in range(n):
        s, e = int(rp[q]), int(rp[q + 1])
        perm = rng.permutation(e - s)
        pre_s[s:e], ww_s[s:e] = pre[s:e][perm], ww[s:e][perm]
    be2 = CudaLatticeBackend(K.MODEL_IZH, 0, 0, rows, cols)
    be2.connect_csr(0, 0, rp, pre_s, ww_s)
    rp2, pre2, ww2 = be2.get_connection_csr()
    assert (rp2 == rp).all() and (pre2 == pre).all() and (ww2 == ww).all()
    assert be2.connection_nnz() == pre.size
    # GraphGPU index_to_position (graph/mod.rs:300-361): a permuted graph index space lands on the same cells
    itp = rng.permutation(n).astype(np.uint32)
    inv = np.argsort(itp)
    be3 = CudaLatticeBackend(K.MODEL_IZH, 0, 0, rows, cols)
    be3.connect_dense(0, 0, conn[np.ix_(itp, itp)], w[np.ix_(itp, itp)], index_to_position=itp)
    c3, w3 = be3.get_connection_dense()
    assert (c3 == conn).all() and (w3 == w).all()
    del inv
    # lookup_weight / None vs Some(0.0)
    a, b = np.argwhere(conn == 1)[0]
    assert be.lookup_weight(a, b) == pytest.approx(float(w[a, b]))
    z = np.argwhere(conn == 0)[0]
    assert be.lookup_weight(z[0], z[1]) is None
    with pytest.raises(S.SnnError) as ei:
        be.lookup_weight(0, n)
    assert ei.value.status == K.SNN_GRAPH_POSTSYNAPTIC_NOT_FOUND
    with pytest.raises(S.SnnError) as ei:
        be.lookup_weight(n, 0)
    assert ei.value.status == K.SNN_GRAPH_PRESYNAPTIC_NOT_FOUND
    with pytest.raises(S.SnnError) as ei:
        be.connect_dense(0, 0, np.zeros((3, 3), np.uint32), np.zeros((3, 3), f32))
    assert ei.value.status == K.SNN_GRAPH_DIMENSIONS_DO_NOT_MATCH
    with pytest.raises(S.SnnError) as ei:
        be.connect_csr(0, 0, np.array([0] * n + [1], np.uint64), np.array([n + 3], np.uint32), np.ones(1, f32))
    assert ei.value.status == K.SNN_GRAPH_PRESYNAPTIC_NOT_FOUND


def test_edit_weight_none_some_none_and_row_access(oracle_lattice_factory):
    """Graph::edit_weight(pre, post, Option<f32>) (graph/mod.rs:208-226) through the C ABI: None -> Some(0.0) -> None on a single
    edge, Some(w) over an existing edge (one word on the device), the doc-test of graph/mod.rs:112-137 replayed, error order, and
    snn_lattice_get_graph_rows == the matching rows of the whole-graph CSR.  Every state is stepped against the oracle."""
    rows, cols = 4, 5
    n = rows * cols

    def make(fac):
        lat = SC.build_lattice(fac, model="izh", rows=rows, cols=cols, seed=3, graph="random", history=False)
        return lat
    a, b = make(None), make(oracle_lattice_factory)
    conn, w = a.graph_dense()
    z = [tuple(x) for x in np.argwhere(conn == 0) if x[0] != x[1]][0]
    e = tuple(np.argwhere(conn == 1)[3])
    pos = lambda i: (int(i) // cols, int(i) % cols)
    for lat in (a, b):
        assert lat.get_weight(pos(z[0]), pos(z[1])) is None
        lat.edit_weight(pos(z[0]), pos(z[1]), 0.0)          # None -> Some(0.0): connected, counted in the averages
        assert lat.get_weight(pos(z[0]), pos(z[1])) == 0.0
        lat.edit_weight(pos(e[0]), pos(e[1]), 1.75)         # Some -> Some: in place
        assert lat.get_weight(pos(e[0]), pos(e[1])) == 1.75
    a.run_lattice(30); b.run_lattice(30)
    SC.compare_lattices(a, b, exact=True, fields=("current_voltage", "w_value", "last_firing_time"))
    (ca, wa), (cb, wb) = a.graph_dense(), b.graph_dense()
    assert (ca == cb).all() and (wa == wb).all() and ca[z] == 1 and wa[z] == 0.0 and wa[e] == 1.75
    for lat in (a, b):
        lat.edit_weight(pos(z[0]), pos(z[1]), None)         # Some(0.0) -> None
        assert lat.get_weight(pos(z[0]), pos(z[1])) is None
        lat.edit_weight(pos(e[0]), pos(e[1]), None)         # an original edge goes away too
        lat.edit_weight(pos(z[0]), pos(z[1]), None)         # None over None: no-op
    a.run_lattice(30); b.run_lattice(30)
    SC.compare_lattices(a, b, exact=True, fields=("current_voltage", "w_value", "last_firing_time"))
    (ca, wa), (cb, wb) = a.graph_dense(), b.graph_dense()
    assert (ca == cb).all() and (wa == wb).all() and ca[z] == 0 and ca[e] == 0
    # row access == rows of the whole CSR
    rp, pre, ww = a._be.get_connection_csr()
    for (r0, r1) in ((0, n), (3, 4), (7, 15), (n - 1, n), (5, 5)):
        rp2, pre2, ww2 = a._be.get_graph_rows(r0, r1)
        s, t = int(rp[r0]), int(rp[r1])
        assert (rp2 == rp[r0:r1 + 1] - rp[r0]).all() and (pre2 == pre[s:t]).all() and (ww2 == ww[s:t]).all()
    # error order: postsynaptic position first (graph/mod.rs:209-214)
    be = a._be
    for args, code in (((0, n, 1.0), K.SNN_GRAPH_POSTSYNAPTIC_NOT_FOUND), ((n, 0, 1.0), K.SNN_GRAPH_PRESYNAPTIC_NOT_FOUND),
                       ((n, n, 1.0), K.SNN_GRAPH_POSTSYNAPTIC_NOT_FOUND)):
        with pytest.raises(S.SnnError) as ei:
            be.edit_weight(*args)
        assert ei.value.status == code
    # the doc-test of AdjacencyMatrix (graph/mod.rs:112-137) on a 1 x 3 lattice: nodes (0,0) (0,1) (0,2)
    g = CudaLatticeBackend(K.MODEL_IZH, 0, 0, 1, 3)
    g.edit_weight(0, 1, 0.5)
    g.edit_weight(2, 1, 1.0)
    assert g.lookup_weight(0, 1) == 0.5 and g.lookup_weight(1, 0) is None
    rp3, pre3, _ = g.get_graph_rows(1, 2)
    assert pre3.tolist() == [0, 2]                            # get_incoming_connections((0,1)) == {(0,0), (1,2)}
    g.edit_weight(0, 1, None)
    assert g.lookup_weight(0, 1) is None and g.get_graph_rows(1, 2)[1].tolist() == [2]


def test_edit_weight_on_stencil_keeps_the_staged_kernels(oracle_lattice_factory):
    """A weight edit (and the weight read-back after STDP) on a set_graph_grid lattice large enough for the window-staged kernel:
    the block is materialised on the host, yet the rebuilt table keeps the generator's uniform layout — results stay those of the
    oracle, before and after an edge is removed."""
    rows, cols = 264, 256

    def make(fac):
        lat = SC.build_lattice(fac, model="izh", rows=rows, cols=cols, seed=4, graph="grid", hetero=False, history=False,
                               chem="approx_ampa", stdp=False, c_m=2.0)
        rng = np.random.default_rng(9)
        lat.set_field("current_voltage", rng.uniform(-65, 30, rows * cols).astype(f32))
        lat.set_field("b", rng.uniform(0.25, 0.36, rows * cols).astype(f32))
        return lat
    a, b = make(None), make(oracle_lattice_factory)
    for lat in (a, b):
        lat.edit_weight((100, 100), (100, 101), 3.0)
        lat.edit_weight((263, 255), (262, 254), 0.25)
    a.run_lattice(12); b.run_lattice(12)
    for name in ("current_voltage", "last_firing_time", "neurotransmitters$t"):
        assert (a.get_field(name) == b.get_field(name)).all(), name
    for lat in (a, b):
        lat.edit_weight((10, 10), (10, 11), None)            # structural: rebuild through the host CSR
        lat.edit_weight((10, 12), (10, 10), 2.0)             # not a stencil edge: added
    a.run_lattice(12); b.run_lattice(12)
    for name in ("current_voltage", "last_firing_time", "neurotransmitters$t"):
        assert (a.get_field(name) == b.get_field(name)).all(), name
    assert a.get_weight((10, 10), (10, 11)) is None and a.get_weight((10, 12), (10, 10)) == 2.0 and a.get_weight((100, 100), (100, 101)) == 3.0


def test_spike_history_aggregate_on_device(oracle_lattice_factory):
    """SpikeHistory::aggregate (neuron/mod.rs:335-359) from the device-side counts, across several run calls and a reset."""
    a = SC.build_lattice(None, model="izh", rows=9, cols=11, seed=5)
    b = SC.build_lattice(oracle_lattice_factory, model="izh", rows=9, cols=11, seed=5)
    assert (a.spike_history.aggregate() == 0).all() and a.spike_history.aggregate().shape == (9, 11)
    for k in (70, 1, 129):
        a.run_lattice(k); b.run_lattice(k)
    agg = a.spike_history.aggregate()
    assert agg.dtype == np.int64 and agg.sum() > 20
    assert (agg == a.spike_history.history.sum(axis=0)).all()
    assert (agg == b.spike_history.aggregate()).all()
    a.spike_history.reset()
    a.run_lattice(40)
    assert (a.spike_history.aggregate() == a.spike_history.history.sum(axis=0)).all()


def test_grid_generator_equals_connect_predicate(oracle_lattice_factory):
    """set_graph_grid(radius) == Lattice::connect(|x,y| max(|dr|,|dc|) <= radius && x != y, None) (neuron/mod.rs:1134-1157)."""
    for radius in (1, 2):
        lat = S.Lattice(S.IzhikevichNeuron)
        lat.populate(S.IzhikevichNeuron(), 5, 6)
        lat.connect_grid(radius, 1.0)
        ref = S.Lattice(S.IzhikevichNeuron, backend_factory=oracle_lattice_factory)
        ref.populate(S.IzhikevichNeuron(), 5, 6)
        ref.connect(lambda x, y: x != y and max(abs(x[0] - y[0]), abs(x[1] - y[1])) <= radius)
        (ca, wa), (cb, wb) = lat.graph_dense(), ref.graph_dense()
        assert (ca == cb).all() and (wa == wb).all()
        assert lat.get_weight((0, 0), (1, 1)) == 1.0 and lat.get_weight((0, 0), (4, 5)) is None


def test_size_zero_and_noop_cases():
    """tests/size_zero_cases.rs: 0x0 lattices return Ok; zero iterations and both synapse flags off are no-ops."""
    for rows, cols in [(0, 0), (0, 4), (3, 0)]:
        lat = S.Lattice(S.IzhikevichNeuron)
        lat.populate(S.IzhikevichNeuron(), rows, cols)
        lat.connect(lambda x, y: True)
        lat.run_lattice(10)
        assert lat.cell_grid() == [[]] * rows or lat.cell_grid() == []
    never = S.Lattice(S.IzhikevichNeuron)
    never.run_lattice(5)
    lat = SC.build_lattice(None, model="izh", rows=3, cols=3, history=False)
    v0 = lat.get_field("current_voltage")
    lat.run_lattice(0)
    assert (lat.get_field("current_voltage") == v0).all() and lat.internal_clock == 0
    lat.electrical_synapse = False
    lat.chemical_synapse = False
    lat.run_lattice(50)
    assert (lat.get_field("current_voltage") == v0).all() and lat.internal_clock == 0
    net = S.LatticeNetwork()
    net.run_lattices(3)


def test_set_cell_grid_dimension_invariant():
    """tests/grid_formation_invariant.rs: set_cell_grid rejects a grid of different dimensions."""
    lat = S.Lattice(S.IzhikevichNeuron)
    lat.populate(S.IzhikevichNeuron(), 2, 3)
    grid = lat.cell_grid()
    with pytest.raises(S.SnnError) as ei:
        lat.set_cell_grid(grid[:1])
    assert ei.value.status == K.SNN_GRAPH_POSITION_NOT_FOUND
    with pytest.raises(S.SnnError):
        lat.set_cell_grid([row[:2] for row in grid])
    grid[1][2].current_voltage = -12.5
    grid[0][1].last_firing_time = 17
    lat.set_cell_grid(grid)
    g2 = lat.cell_grid()
    assert g2[1][2].current_voltage == -12.5 and g2[0][1].last_firing_time == 17 and g2[0][0].last_firing_time is None


def test_apply_and_timing_controls():
    lat = S.Lattice(S.IzhikevichNeuron)
    lat.populate(S.IzhikevichNeuron(gap_conductance=10.0), 3, 3)
    lat.apply(lambda nrn: setattr(nrn, "current_voltage", 29.99))
    lat.apply_given_position(lambda pos, nrn: setattr(nrn, "d", float(pos[0] * 3 + pos[1])))
    assert (lat.get_field("d") == np.arange(9, dtype=f32)).all()
    lat.connect_grid()
    lat.run_lattice(1)
    assert (lat.get_field("last_firing_time") == 0).all() and lat.internal_clock == 1
    assert (lat.get_field("is_spiking") == 1).all()
    lat.run_lattice(2)
    assert lat.internal_clock == 3
    lat.reset_timing()
    assert lat.internal_clock == 0 and (lat.get_field("last_firing_time") == -1).all()
    lat.set_dt(0.05)
    assert (lat.get_field("dt") == f32(0.05)).all() and lat.plasticity.dt == 0.05
    assert lat._be.get_plasticity()[4] == pytest.approx(0.05)


def test_network_error_codes_and_ids():
    """LatticeNetwork::add_lattice / connect error behaviour (neuron/mod.rs:1663-1698, 1852-1862)."""
    be = CudaNetworkBackend(K.MODEL_IZH)
    be.add_lattice(1, 2, 2)
    be.add_train_lattice(0, 1, 2)
    with pytest.raises(S.SnnError) as ei:
        be.add_lattice(1, 3, 3)
    assert ei.value.status == K.SNN_NET_GRAPH_ID_ALREADY_PRESENT
    with pytest.raises(S.SnnError) as ei:
        be.add_train_lattice(1, 1, 1)
    assert ei.value.status == K.SNN_NET_GRAPH_ID_ALREADY_PRESENT
    lib, h = be.lib, be.h
    c, w = np.ones(4, np.uint32), np.ones(4, f32)
    assert lib.snn_network_connect_dense(h, 1, 0, c.ctypes.data, w.ctypes.data, 4, 2) == K.SNN_NET_POSTSYNAPTIC_LATTICE_CANNOT_BE_SPIKE_TRAIN
    assert lib.snn_network_connect_dense(h, 7, 1, c.ctypes.data, w.ctypes.data, 4, 4) == K.SNN_NET_PRESYNAPTIC_ID_NOT_FOUND
    assert lib.snn_network_connect_dense(h, 1, 9, c.ctypes.data, w.ctypes.data, 4, 4) == K.SNN_NET_POSTSYNAPTIC_ID_NOT_FOUND
    assert lib.snn_network_connect_dense(h, 0, 1, c.ctypes.data, w.ctypes.data, 3, 4) == K.SNN_GRAPH_DIMENSIONS_DO_NOT_MATCH
    be.connect_dense(0, 1, np.ones((2, 4), np.uint32), np.full((2, 4), 0.25, f32))
    assert be.connection_nnz(0, 1) == 8
    # fields set before a later lattice is added survive the re-layout
    be.set_field(1, "current_voltage", [1.0, 2.0, 3.0, 4.0])
    be.add_lattice(0 + 5, 3, 3)
    be.add_train_lattice(3, 2, 2)
    assert (be.get_field(1, "current_voltage") == f32([1, 2, 3, 4])).all()
    c2, w2 = be.get_connection_dense(0, 1)
    assert (c2 == 1).all() and (w2 == 0.25).all()


def test_spike_train_lattice_alone_and_rate_kat():
    """RunSpikeTrainLattice (neuron/mod.rs:1419-1428) + tests/rate_spike_train.rs:54-72 on the device."""
    st = S.SpikeTrainLattice(S.RateSpikeTrain, id=4)
    st.populate(S.RateSpikeTrain(rate=100.0, dt=1.0), 2, 3)
    st.update_spike_history = True
    st.run_lattice(1001)
    s = st.spike_history.history.reshape(1001, 6)
    for i in range(1001):
        assert bool(s[i].all()) == bool(s[i].any()) == (i != 0 and (i + 1) % 100 == 0)
    assert (st.get_field("last_firing_time") == 999).all() and st.internal_clock == 1001
    cells = st.spike_train_grid()
    assert cells[0][0].rate == 100.0 and cells[1][2].last_firing_time == 999


def test_plasticity_variant_error_behaviour():
    """BCM / reward-modulation entry points: argument checks and scope limits (no abort, status + last-error string)."""
    import ctypes as C
    izh = CudaLatticeBackend(K.MODEL_IZH, 0, 0, 4, 4)
    b = K.BcmStruct(0.1, 0.1, 0.1)
    assert izh.lib.snn_lattice_set_bcm_plasticity(izh.h, 1, C.byref(b)) == K.SNN_INVALID_ARGUMENT   # neurons without BCMActivity
    assert b"BCMActivity" in izh.lib.snn_lattice_last_error(izh.h)
    r = np.zeros(3, f32)
    assert izh.lib.snn_lattice_run_with_rewards(izh.h, r.ctypes.data, 3) == K.SNN_INVALID_ARGUMENT   # not a reward-modulated lattice
    assert izh.lib.snn_lattice_get_connection_traces(izh.h, None, None, None, 0) == K.SNN_INVALID_ARGUMENT
    izh.connect_grid(0, 1, 1.0)
    izh.set_reward_modulator(True, True, dopamine=0.0, tau_d=20.0, tau_c=1e-4, a_plus=2.0, a_minus=2.0, tau_plus=4.5, tau_minus=4.5, dt=0.1)
    assert izh.lib.snn_lattice_get_connection_traces(izh.h, None, None, None, 5) == K.SNN_SIZE_MISMATCH
    cnt, dw, c = izh.connection_traces()
    assert cnt.size == izh.connection_nnz() == 84 and not cnt.any() and not dw.any() and not c.any()   # TraceRSTDP::default
    izh.run_with_rewards([])                      # zero iterations: Ok(())
    assert izh.get_option(K.OPT_INTERNAL_CLOCK) == 0
    izh.run_with_rewards([0.5, -0.25])
    assert izh.get_option(K.OPT_INTERNAL_CLOCK) == 2
    d = izh.get_reward_modulator()["dopamine"]
    want = f32(f32(f32(0) * np.exp(f32(-0.1) / f32(20))) + f32(20) * f32(0.5))
    want = f32(f32(want * np.exp(f32(-0.1) / f32(20), dtype=f32)) + f32(20) * f32(-0.25))
    assert d == pytest.approx(float(want), rel=1e-6)
    # networks are out of scope this round (row-strip partitioned lattices are covered by tests/mgpu_parity.py --reward)
    net = CudaNetworkBackend(K.MODEL_IZH)
    assert not hasattr(net, "set_reward_modulator")


@pytest.mark.parametrize("case", ["izh_grid_hist", "hh_chem", "lif_stdp_random", "net_rate_stdp", "net_preset_wide", "net_poisson"])
def test_multi_step_launch_is_bit_identical_to_one_launch_per_step(case):
    """SNN_OPT_STEPS_PER_GRAPH: 0 = the whole run inside one cooperative launch (step_multi.cu, grid-wide barrier between
    timesteps), 1 = one launch per timestep, 7 = at most seven per launch.  Same arithmetic in the same order: every field, every
    history record and every weight must be bit-identical, including odd step counts (ping-pong parity), several run calls
    (pending STDP across launches) and networks whose spike trains step between the neurons of consecutive timesteps."""
    import test_gpu_parity as TP

    def build():
        if case == "izh_grid_hist":
            return SC.build_lattice(None, model="izh", rows=37, cols=41, seed=3, graph="grid"), None
        if case == "hh_chem":
            return SC.build_lattice(None, model="hh", rows=19, cols=23, seed=4, graph="grid2", chem="destexhe_all", gap=2.0), None
        if case == "lif_stdp_random":
            return SC.build_lattice(None, model="lif", rows=9, cols=12, seed=5, graph="random", stdp=True, gap=40.0), None
        if case == "net_rate_stdp":
            return None, TP.build_network(None, None, train="rate", stdp=True)
        if case == "net_preset_wide":
            return None, TP.build_network(None, None, train="preset", stdp=True, st_shape=(8, 9))
        net = TP.build_network(None, None, train="poisson", stdp=True)
        net._be.set_option(K.OPT_RNG_SEED, 77)
        return None, net

    results = []
    for spg in (1, 0, 7):
        lat, net = build()
        be = (lat or net)._be
        be.set_option(K.OPT_STEPS_PER_GRAPH, spg)
        assert be.get_option(K.OPT_STEPS_PER_GRAPH) == spg
        launches = 0
        for k in (33, 1, 50):
            if lat is not None:
                lat._push_options()
            else:
                net.run_lattices(0)   # pushes the options
            ms, nl = be.run_timed(k)
            launches += nl
        out = {"launches": launches}
        if lat is not None:
            for name in SC.lattice_field_names(lat):
                out[name] = lat.get_field(name)
            out["grid"], out["spikes"] = lat.grid_history.history, lat.spike_history.history
            out["w"] = lat.graph_csr()[2]
        else:
            for lid in (1, 2):
                L = net.get_lattice(lid)
                for name in SC.lattice_field_names(L):
                    out[f"{lid}/{name}"] = L.get_field(name)
                out[f"{lid}/grid"], out[f"{lid}/spikes"] = L.grid_history.history, L.spike_history.history
            st = net.get_spike_train_lattice(0)
            out["st/spikes"] = st.spike_history.history
            out["st/lft"] = st.get_field("last_firing_time")
            for pre, post in TP.PAIRS:
                out[f"w{pre}{post}"] = net._be.get_connection_dense(pre, post)[1]
        results.append(out)
    one, whole, seven = results
    assert whole["launches"] < one["launches"] / 10, (whole["launches"], one["launches"])
    assert whole["launches"] < seven["launches"] < one["launches"]
    for key in one:
        if key == "launches":
            continue
        for other, label in ((whole, "whole-run launch"), (seven, "7 steps per launch")):
            a, b = np.asarray(one[key]), np.asarray(other[key])
            assert a.shape == b.shape and (a.view(np.uint8) == b.view(np.uint8)).all() if a.dtype != bool else (a == b).all(), (key, label)
    if case in ("izh_grid_hist", "net_rate_stdp", "net_preset_wide", "net_poisson"):
        spikes = one["spikes"].sum() if "spikes" in one else one["1/spikes"].sum() + one["2/spikes"].sum()
        assert spikes > 0
