"""Spike events (SNN_OPT_UPDATE_SPIKE_EVENTS): per lattice and recorded step, the flat indices of the cells that spiked, compacted
on the device from the staged spike raster.  The events are the same data as the dense SpikeHistory raster: every check compares
them with np.nonzero of that raster (or of another handle's), exactly.

CPU tier: the oracle through the front end (it answers the event calls from its dense raster), and the rank merge of
snn_b200.dist, in process and over gloo.  GPU tier: the device against its own dense history on every step path, across
history chunks, with events only, on partitions, and recording against not recording."""
import os
import socket
import subprocess
import sys
import textwrap

import ctypes as C
import numpy as np
import pytest

import scenarios as SC
import snn_b200 as S
from oracle_api import OracleBackend
from snn_b200 import _capi as K
from snn_b200.backend import CudaLatticeBackend
from snn_b200.dist import LocalStrips, merge_spike_events
from test_gpu_parity import build_network

f32 = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class EventsOracle(OracleBackend):
    """The CPU oracle answering the spike-event calls from its dense raster, which records while either option is on."""

    def __init__(self, *a, **kw):
        self._events = {}
        super().__init__(*a, **kw)

    def _apply(self, lid):
        fl = self._flags[lid]
        self._ck(self.L.orc_set_lattice_flags(self.h, lid, fl[0], fl[1], int(fl[2] or self._events.get(lid, 0))))

    def set_option(self, option, value, id=None):
        lid = 0 if id is None else id
        if option == K.OPT_UPDATE_SPIKE_EVENTS:
            self._events[lid] = int(value)
            self._apply(lid)
            return
        super().set_option(option, value, id)
        if option == K.OPT_UPDATE_SPIKE_HISTORY:
            self._apply(lid)

    def spike_events(self, id=0):
        h = self.spike_history(id)
        steps, neurons = np.nonzero(h)
        step_ptr = np.zeros(h.shape[0] + 1, np.uint64)
        step_ptr[1:] = np.cumsum(np.bincount(steps, minlength=h.shape[0]))
        return step_ptr, neurons.astype(np.uint32)


@pytest.fixture
def ev_lattice_factory():
    return lambda model, ntk, rck, rows, cols: EventsOracle(model, ntk, rck, rows=rows, cols=cols)


@pytest.fixture
def ev_network_factory():
    return lambda model, ntk, rck, tk, rf: EventsOracle(model, ntk, rck, tk, rf)


def _check_against_dense(owner, steps=None):
    """owner.spike_events against np.nonzero of owner.spike_history, exactly; returns the number of events."""
    ev = owner.spike_events
    dense = owner.spike_history.history.reshape(ev.steps if steps is None else steps, -1)
    assert ev.steps == dense.shape[0]
    want = np.argwhere(dense)
    assert ev.pairs().shape == want.shape and (ev.pairs() == want).all()
    assert (ev.step_ptr[1:] - ev.step_ptr[:-1] == dense.sum(axis=1)).all()
    assert (ev.dense() == owner.spike_history.history).all()
    return ev.neurons.size


# ------------------------------------------------------------------ CPU tier
@pytest.mark.parametrize("model,graph,stdp", [("izh", "grid", True), ("qif", "csr", False)])
def test_oracle_events_equal_the_dense_raster(model, graph, stdp, ev_lattice_factory):
    lat = SC.build_lattice(ev_lattice_factory, model=model, rows=7, cols=9, seed=5, graph=graph, stdp=stdp)
    lat.update_spike_events = True
    for k in (11, 6):
        lat.run_lattice(k)
        assert _check_against_dense(lat) > 0
    lat.spike_history.reset()
    assert lat.spike_events.steps == 0 and lat.spike_events.neurons.size == 0


def test_oracle_network_events_equal_the_dense_raster(ev_lattice_factory, ev_network_factory):
    net = build_network(ev_lattice_factory, ev_network_factory, train="rate")
    for lid in (1, 2):
        net.get_lattice(lid).update_spike_events = True
    net.get_spike_train_lattice(0).update_spike_events = True
    net.run_lattices(36)
    for owner in (net.get_lattice(1), net.get_lattice(2), net.get_spike_train_lattice(0)):
        assert _check_against_dense(owner) > 0


def test_merge_concatenates_the_ranks_step_by_step():
    rows, cols = 5, 4
    rng = np.random.default_rng(2)
    dense = rng.random((6, rows * cols)) < 0.3
    bounds = [0, 2, 3, 5]
    parts = []
    for r in range(3):
        sub = dense[:, bounds[r] * cols:bounds[r + 1] * cols]
        steps, idx = np.nonzero(sub)
        sp = np.zeros(7, np.uint64)
        sp[1:] = np.cumsum(sub.sum(axis=1))
        parts.append((sp, (idx + bounds[r] * cols).astype(np.uint32)))
    ev = merge_spike_events(parts, rows, cols)
    assert (ev.pairs() == np.argwhere(dense)).all()
    assert (ev.dense().reshape(6, -1) == dense).all()
    with pytest.raises(ValueError):
        merge_spike_events([parts[0], (parts[1][0][:-1], parts[1][1][:0])], rows, cols)


GLOO_WORKER = textwrap.dedent('''
    import os, sys
    import numpy as np
    import torch.distributed as dist
    sys.path[:0] = [os.path.join(ROOT, "spiking-neural-networks_b200")]
    from snn_b200.dist import gather_spike_events, partition_rows

    dist.init_process_group("gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    rows, cols, steps = 9, 6, 12
    dense = np.random.default_rng(4).random((steps, rows * cols)) < 0.25
    r0, r1 = partition_rows(rows, world, rank)

    class Rank:   # the two calls gather_spike_events makes on a partitioned lattice back end
        def spike_events(self):
            sub = dense[:, r0 * cols:r1 * cols]
            s, idx = np.nonzero(sub)
            sp = np.zeros(steps + 1, np.uint64)
            sp[1:] = np.cumsum(sub.sum(axis=1))
            return sp, (idx + r0 * cols).astype(np.uint32)

        def shape(self):
            return r1 - r0, cols

    ev = gather_spike_events(Rank(), rank, world)
    assert (ev.rows, ev.cols) == (rows, cols)
    assert (ev.pairs() == np.argwhere(dense)).all()
    print("GLOO_EVENTS_OK")
    dist.destroy_process_group()
''')


def test_gather_spike_events_over_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(f"ROOT = {ROOT!r}\n" + GLOO_WORKER)
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "3", "--master-addr", "127.0.0.1",
           "--master-port", str(port), str(script)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=dict(os.environ, OMP_NUM_THREADS="1"))
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    assert res.stdout.count("GLOO_EVENTS_OK") == 3


# ------------------------------------------------------------------ GPU tier
@pytest.fixture(params=["auto", "tma", "tma_l1"])
def kernel_path(request, monkeypatch):
    """The automatic kernel choice, the TMA-staged kernels forced where eligible, and the window kernel off (as in
    tests/test_gpu_parity.py)."""
    monkeypatch.setenv("SNN_B200_TMA", "1" if request.param == "auto" else "2")
    monkeypatch.setenv("SNN_B200_WIN", "0" if request.param == "tma_l1" else "1")
    return request.param


LATTICES = {   # (build_lattice keywords, BCM rule, run lengths: odd and even)
    "izh": (dict(model="izh", graph="grid"), False, (7, 10, 1, 4)),
    "izh_csr": (dict(model="izh", graph="csr"), False, (7, 10, 1, 4)),
    "lif_stdp": (dict(model="lif", graph="grid", stdp=True), False, (7, 10, 1, 4)),
    # AMPA, NMDA and GABA; this lattice first spikes after about 420 steps
    "hh_chem": (dict(model="hh", graph="grid", chem="destexhe_all", gap=SC.drive_current("hh")), False, (301, 150, 1, 48)),
    "bcm_izh": (dict(model="bcm_izh", graph="grid", stdp=True), True, (7, 10, 1, 4)),
}


def _device_lattice(kind, rows=20, cols=24, seed=3, **over):
    kw, bcm, _ = LATTICES[kind]
    lat = SC.build_lattice(None, rows=rows, cols=cols, seed=seed, **{**kw, **over})
    if bcm:
        lat.plasticity = S.BCM(decay=0.05, average_scalar=0.5, dt=1e-6)
    return lat


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(LATTICES))
def test_events_equal_the_dense_history_on_every_kernel_path(kind, kernel_path):
    lat = _device_lattice(kind)
    lat.update_spike_events = True
    done = 0
    for k in LATTICES[kind][2]:
        lat.run_lattice(k)
        done += k
        n = _check_against_dense(lat)
        assert lat.spike_events.steps == done
    assert n > 0


@pytest.mark.gpu
@pytest.mark.parametrize("steps_per_graph", [0, 1])
def test_events_with_the_multi_step_kernel(steps_per_graph):
    lat = _device_lattice("izh_csr", rows=9, cols=11)
    lat.update_spike_events = True
    lat._be.set_option(K.OPT_STEPS_PER_GRAPH, steps_per_graph)
    for k in (9, 14, 3):
        lat.run_lattice(k)
    assert _check_against_dense(lat) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("st_shape", [(3, 4), (8, 9)])
def test_network_events_of_neuron_and_spike_train_lattices(st_shape):
    net = build_network(None, None, train="rate", st_shape=st_shape)
    for lid in (1, 2):
        net.get_lattice(lid).update_spike_events = True
    net.get_spike_train_lattice(0).update_spike_events = True
    for k in (15, 20, 1):
        net.run_lattices(k)
    for owner in (net.get_lattice(1), net.get_lattice(2), net.get_spike_train_lattice(0)):
        assert _check_against_dense(owner) > 0


@pytest.mark.gpu
def test_events_across_history_chunks_and_events_only():
    """1000 x 1024 neurons with the grid history on stage 64 steps per 256 MiB chunk: 150 steps span three chunks (the event
    buffer grows when a later chunk holds more events).  Events alone stage 2048 steps per chunk: one chunk, the same events."""
    kw = dict(model="izh", rows=1000, cols=1024, seed=8, graph="grid", history=False)
    both, only = SC.build_lattice(None, **kw), SC.build_lattice(None, **kw)
    both.update_grid_history = both.update_spike_history = both.update_spike_events = True
    only.update_spike_events = True
    for lat in (both, only):
        lat.run_lattice(150)
    assert _check_against_dense(both, 150) > 0
    a, b = both.spike_events, only.spike_events
    assert (a.step_ptr == b.step_ptr).all() and (a.neurons == b.neurons).all()
    assert only._be.history_len() == 0 and only.spike_history.history.shape[0] == 0


def _strip_fields(n, seed):
    rng = np.random.default_rng(seed)
    return {"current_voltage": rng.uniform(-65, 30, n).astype(f32), "b": rng.uniform(0.25, 0.36, n).astype(f32),
            "gap_conductance": (10 * rng.uniform(0.5, 1.5, n)).astype(f32), "c_m": np.full(n, 2.0, f32)}


@pytest.mark.gpu
@pytest.mark.parametrize("world,general", [(2, False), (3, False), (2, True), (3, True), (4, True)])
def test_partition_events_equal_the_whole_lattice(world, general):
    rows, cols = 27, 16
    n = rows * cols
    fields = _strip_fields(n, 11 + world)
    whole = CudaLatticeBackend(K.MODEL_IZH, 0, 0, rows, cols)
    parts = LocalStrips(K.MODEL_IZH, rows, cols, world)
    for name, a in fields.items():
        whole.set_field(0, name, a)
        parts.set_field(name, a)
    if general:
        conn, w = SC.random_graph(rows, cols, 31, radius=6.0, p=0.3, weights="rand")
        rp, pre, ww = SC.dense_to_csr(conn, w)
        whole.connect_csr(0, 0, rp, pre, ww)
        parts.set_graph_csr(rp, pre, ww)
        parts.attach_general()
    else:
        whole.connect_grid(0, 1, 1.0)
        parts.each(lambda be: be.connect_grid(0, 1, 1.0))
        parts.attach()
    for be in [whole] + parts.strips:
        be.set_option(K.OPT_ELECTRICAL_SYNAPSE, 1)
        be.set_option(K.OPT_UPDATE_SPIKE_EVENTS, 1, 0)
    for k in (9, 6):
        parts.run(k)
        whole.run(k)
    sp, nr = whole.spike_events()
    merged = parts.spike_events()
    assert nr.size > 0 and (merged.step_ptr == sp).all() and (merged.neurons == nr).all()
    for r, be in enumerate(parts.strips):
        own = parts.rows_of(r)
        _, idx = be.spike_events()
        assert ((idx >= own.start) & (idx < own.stop)).all()


@pytest.mark.gpu
def test_recording_does_not_perturb_the_run():
    kw = dict(model="izh", rows=40, cols=50, seed=9, graph="grid", stdp=True, history=True)
    on, never = SC.build_lattice(None, **kw), SC.build_lattice(None, **kw)
    on.update_spike_events = True
    for k in (13, 8):
        on.run_lattice(k)
        never.run_lattice(k)
        for nm in ("current_voltage", "w_value", "last_firing_time"):
            assert (on.get_field(nm) == never.get_field(nm)).all(), nm
        assert (on.spike_history.history == never.spike_history.history).all()
        assert (on.graph_csr()[2] == never.graph_csr()[2]).all()
    on.update_spike_events = False
    on._push_options()
    assert on._be.run_timed(6)[1] == never._be.run_timed(6)[1]


@pytest.mark.gpu
def test_reset_rules_and_capacity():
    lat = _device_lattice("izh")
    lat.update_spike_events = True
    lat.run_lattice(12)
    steps, n = C.c_uint64(), C.c_uint64()
    lib, h = lat._be.lib, lat._be.h
    assert lib.snn_lattice_spike_event_count(h, C.byref(steps), C.byref(n)) == K.SNN_OK and n.value > 0
    lat.reset_timing()
    assert lat.spike_events.steps == 12 and lat.spike_events.neurons.size == n.value
    sp = np.zeros(steps.value + 1, np.uint64)
    small = np.zeros(n.value - 1, np.uint32)
    st = lib.snn_lattice_get_spike_events(h, sp.ctypes.data_as(C.c_void_p), small.ctypes.data_as(C.c_void_p), small.size)
    dense = np.zeros(12 * lat.size - 1, np.uint8)
    assert st == lib.snn_lattice_get_spike_history(h, dense.ctypes.data_as(C.c_void_p), dense.size) == K.SNN_SIZE_MISMATCH
    lat.spike_history.reset()
    assert lat.spike_events.steps == 0 and lat.spike_events.neurons.size == 0
    lat.run_lattice(3)
    assert _check_against_dense(lat) >= 0 and lat.spike_events.steps == 3
