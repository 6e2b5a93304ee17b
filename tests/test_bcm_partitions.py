"""BCM plasticity on row strips and general-graph partitions, every partition a handle of this process on ONE GPU
(snn_lattice_attach_local / gpart_attach_local).  An edge whose presynaptic neuron lives on another rank is updated by the rank that
owns its postsynaptic row, from the spike time and current_activity the neighbour exported after the step.  Per edge that is the
same arithmetic in the same order as on the whole lattice, and BCM calls no transcendental function: the partitions must match
the whole lattice on one GPU and the CPU oracle bit for bit."""
import threading

import numpy as np
import pytest

import scenarios as SC
import snn_b200 as S
from snn_b200 import _capi as K
from snn_b200.backend import CudaLatticeBackend
from snn_b200.dist import LocalStrips
from oracle_api import OracleBackend

pytestmark = pytest.mark.gpu
f32 = np.float32

BCM = dict(decay=0.05, average_scalar=0.5, dt=1e-6)   # the parameters of the whole-lattice BCM tests
STATE = ["current_voltage", "w_value", "last_firing_time", "is_spiking"]
BOOKKEEPING = ["average_activity", "current_activity", "num_spikes", "firing_rate_clock", "period"]


def _fields(n, seed, chem):
    """Per-neuron fields of a tonically firing BCM Izhikevich lattice (the recipe of scenarios.build_lattice)."""
    rng = np.random.default_rng(seed)
    fl = {"current_voltage": (rng.uniform(-65, 30, n).astype(f32), 1),
          "gap_conductance": ((10 * rng.uniform(0.5, 1.5, n)).astype(f32), 1),
          "firing_rate_window": (rng.choice([1.5, 2.0, 3.25], n).astype(f32), 1),
          "period": (rng.choice([2, 3, 5], n).astype(np.uint32), 1),
          "a": (rng.uniform(0.015, 0.03, n).astype(f32), 1),
          "b": (rng.uniform(0.25, 0.36, n).astype(f32), 1),
          "d": (rng.uniform(6.0, 9.0, n).astype(f32), 1),
          "c_m": (np.full(n, 2.0, f32), 1)}
    if chem:
        flags = np.zeros((n, 3), np.uint32)
        flags[:, 0] = 1
        fl["neurotransmitters$flags"] = (flags, 3)
        fl["receptors$flags"] = (flags, 3)
    return fl


def _options(be, chem):
    be.set_option(K.OPT_ELECTRICAL_SYNAPSE, 1)
    be.set_option(K.OPT_CHEMICAL_SYNAPSE, int(bool(chem)))
    be.set_option(K.OPT_DO_PLASTICITY, 1, 0)


def _bcm(be):
    be.set_bcm_plasticity(0, True, BCM["decay"], BCM["average_scalar"], BCM["dt"])


def _whole(backend, rows, cols, seed, chem, graph):
    """The same lattice as one handle: the CPU oracle or the device."""
    be = backend(rows, cols)
    for name, (a, _) in _fields(rows * cols, seed, chem).items():
        be.set_field(0, name, a.reshape(-1))
    if graph[0] == "grid":
        be.connect_grid(0, graph[1], 0.8)
    else:
        be.connect_csr(0, 0, *graph[1:])
    _options(be, chem)
    _bcm(be)
    return be


def _oracle(rows, cols):
    return OracleBackend(K.MODEL_BCM_IZH, 0, 0, rows=rows, cols=cols)


def _device(rows, cols):
    return CudaLatticeBackend(K.MODEL_BCM_IZH, 0, 0, rows, cols)


def _strips(rows, cols, world, seed, chem, graph, bcm_after_attach):
    parts = LocalStrips(K.MODEL_BCM_IZH, rows, cols, world)
    for name, (a, per) in _fields(rows * cols, seed, chem).items():
        parts.set_field(name, a, per)
    if graph[0] == "grid":
        parts.each(lambda be: be.connect_grid(0, graph[1], 0.8))
    else:
        parts.set_graph_csr(*graph[1:])
    parts.each(lambda be: _options(be, chem))
    if not bcm_after_attach:
        parts.each(_bcm)
    parts.attach() if graph[0] == "grid" else parts.attach_general()
    if bcm_after_attach:   # the model fixes the slab layout at create time: BCM can be switched on at any point before run
        parts.each(_bcm)
    return parts


def _rank_of_node(parts, n):
    rank = np.zeros(n, np.int64)
    for r in range(parts.world):
        rank[parts.rows_of(r)] = r
    return rank


def _check(parts, ob, dev, runs, rows, cols):
    """Step the partitions, the oracle and the whole device lattice side by side; compare after every run call, bit for bit."""
    n = rows * cols
    w0 = ob.get_connection_csr()[2].copy()
    done = 0
    for k in runs:
        parts.run(k)
        ob.run(k)
        dev.run(k)
        done += k
        for nm in STATE + BOOKKEEPING:
            got, want, whole = parts.get_field(nm), ob.get_field(0, nm), dev.get_field(0, nm)
            assert (whole == want).all(), f"whole lattice: {nm} after {done} steps"
            assert (got == want).all(), f"partitions: {nm} after {done} steps ({int((got != want).sum())} of {got.size})"
        rp, pre, w = parts.graph_csr()
        orp, opre, ow = ob.get_connection_csr()
        assert (rp == orp).all() and (pre == opre).all()
        assert (dev.get_connection_csr()[2] == ow).all(), f"whole lattice: weights after {done} steps"
        assert (w == ow).all(), f"partitions: weights after {done} steps ({int((w != ow).sum())} of {w.size})"
    assert (ob.get_field(0, "last_firing_time") >= 0).sum() > n // 4
    # the boundary really carried the update: edges whose presynaptic neuron lives on another rank and has spiked
    rank = _rank_of_node(parts, n)
    post = np.repeat(np.arange(n), np.diff(orp.astype(np.int64)))
    spiked = ob.get_field(0, "last_firing_time") >= 0
    cross = (rank[post] != rank[opre]) & spiked[opre]
    moved = cross & (ow != w0)
    assert cross.sum() > 0 and moved.sum() >= cross.sum() // 2, (int(cross.sum()), int(moved.sum()))
    assert (w[cross] == ow[cross]).all()
    return cross.sum()


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("shape,radius,chem,after", [((29, 18), 1, None, False), ((31, 16), 2, None, True),
                                                     ((27, 20), 1, "ampa", True), ((33, 14), 2, "ampa", False)])
def test_bcm_strips_match_the_oracle_bit_for_bit(world, shape, radius, chem, after):
    rows, cols = shape
    graph = ("grid", radius)
    parts = _strips(rows, cols, world, 31, chem, graph, after)
    _check(parts, _whole(_oracle, rows, cols, 31, chem, graph), _whole(_device, rows, cols, 31, chem, graph), (31, 1, 30), rows, cols)


@pytest.mark.parametrize("kernel", ["win", "tma"])
def test_bcm_strips_staged_kernels(kernel, monkeypatch):
    """Strips large enough for the staged step kernels (2 x 132 x 256, the shape of the window-kernel strip test), forced at this
    size: the window kernel, and the TMA kernel with the window kernel switched off.  Electrical + AMPA."""
    monkeypatch.setenv("SNN_B200_TMA", "2")
    monkeypatch.setenv("SNN_B200_WIN", "1" if kernel == "win" else "0")
    rows, cols, world = 2 * 132, 256, 2
    graph = ("grid", 1)
    parts = _strips(rows, cols, world, 23, "ampa", graph, False)
    parts.each(lambda be: be.set_option(K.OPT_HALO_TIMEOUT_MS, 20000))
    _check(parts, _whole(_oracle, rows, cols, 23, "ampa", graph), _whole(_device, rows, cols, 23, "ampa", graph), (13, 12), rows, cols)


@pytest.mark.parametrize("world", [2, 3, 4])
@pytest.mark.parametrize("shape,radius,chem", [((12, 9), 2.5, None), ((16, 10), 5.0, "ampa"), ((14, 7), 30.0, None)])
def test_bcm_general_graph_partition_matches_the_oracle_bit_for_bit(world, shape, radius, chem):
    """Random-radius graphs whose edges cross rank boundaries anywhere (radius 30: every rank reads nodes of every other rank,
    also of non-neighbouring ranks): gather-list ghosts, per-neuron export lists, completion counters."""
    rows, cols = shape
    conn, w = SC.random_graph(rows, cols, 41, radius=radius, p=0.6, weights="rand")
    graph = ("csr",) + tuple(SC.dense_to_csr(conn, w))
    parts = _strips(rows, cols, world, 19, chem, graph, world == 3)
    _check(parts, _whole(_oracle, rows, cols, 19, chem, graph), _whole(_device, rows, cols, 19, chem, graph), (21, 1, 20), rows, cols)
    if radius >= 30 and world >= 3:
        assert parts.strips[0].gpart_wants(world - 1)[0].size > 0


def test_bcm_refused_on_a_partition_of_another_model():
    """A partitioned Izhikevich handle has no BCMActivity: SNN_INVALID_ARGUMENT, and the handle keeps stepping with STDP."""
    rows, cols = 20, 16
    n = rows * cols
    parts = LocalStrips(K.MODEL_IZH, rows, cols, 2)
    ob = OracleBackend(K.MODEL_IZH, 0, 0, rows=rows, cols=cols)
    rng = np.random.default_rng(3)
    init = {"current_voltage": rng.uniform(-65, 30, n).astype(f32), "b": rng.uniform(0.25, 0.36, n).astype(f32),
            "c_m": np.full(n, 4.0, f32)}
    for nm, a in init.items():
        parts.set_field(nm, a)
        ob.set_field(0, nm, a)

    def opts(be):
        be.connect_grid(0, 1, 0.8)
        be.set_option(K.OPT_DO_PLASTICITY, 1, 0)
    parts.each(opts)
    opts(ob)
    parts.attach()
    parts.run(9)
    ob.run(9)
    before = {nm: parts.get_field(nm) for nm in STATE}
    w_before = parts.graph_csr()[2]
    for be in parts.strips:
        with pytest.raises(S.SnnError) as ei:
            _bcm(be)
        assert ei.value.status == K.SNN_INVALID_ARGUMENT
    for nm in STATE:
        assert (parts.get_field(nm) == before[nm]).all(), nm
    assert (parts.graph_csr()[2] == w_before).all()
    parts.run(10)
    ob.run(10)
    assert (parts.get_field("last_firing_time") == ob.get_field(0, "last_firing_time")).all()
    np.testing.assert_allclose(parts.graph_csr()[2], ob.get_connection_csr()[2], rtol=1e-4, atol=1e-5)


def test_bcm_strip_launches_one_edge_kernel_per_step():
    """run_timed(k) on a BCM strip: the halo push, k step kernels and k BCM edge kernels; without plasticity the same minus k."""
    rows, cols = 20, 16
    parts = _strips(rows, cols, 2, 5, None, ("grid", 1), False)

    def launches(k):
        out = [None] * parts.world

        def work(r):
            out[r] = parts.strips[r].run_timed(k)[1]
        ts = [threading.Thread(target=work, args=(r,)) for r in range(parts.world)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        assert out[0] == out[1]
        return out[0]
    for k in (1, 5):
        parts.each(lambda be: be.set_option(K.OPT_DO_PLASTICITY, 0, 0))
        plain = launches(k)
        parts.each(lambda be: be.set_option(K.OPT_DO_PLASTICITY, 1, 0))
        assert plain == 1 + k
        assert launches(k) == plain + k
