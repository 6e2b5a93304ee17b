"""Reference-shaped front end: Lattice / SpikeTrainLattice / LatticeNetwork over the C ABI.

Mirrors the reference's public surface for the stepping path (names, argument meaning, error
behaviour): `Lattice::{populate, connect, apply, apply_given_position, set_dt, reset_timing, cell_grid,
set_cell_grid}` + `RunLattice::run_lattice` (neuron/mod.rs:634-700, 1105-1157, 1209-1219),
`LatticeNetwork::{generate_network, add_lattice, add_spike_train_lattice, connect, get_lattice, set_dt,
reset_timing}` + `RunNetwork::run_lattices` (neuron/mod.rs:1612-1930, 2667-2674), and the pub flags
`electrical_synapse, chemical_synapse, do_plasticity, update_grid_history, parallel, internal_clock`
(neuron/mod.rs:556-587).  State lives on the device; host objects are materialised on demand
(`cell_grid()`), which is what `LatticeGPU` does at the end of every run
(gpu_lattices/mod.rs:883-893).
"""
from __future__ import annotations

import numpy as np

from . import _capi as K
from .neurons import (NEURON_CLASSES, NT_KINETICS, RC_KINETICS, RECEPTORS, STDP, IonotropicNeurotransmitterType,
                      IzhikevichNeuron, Neuron, PoissonNeuron, SpikeTrain, RewardModulatedSTDP, BCM)

_NT_PARAM_FIELDS = {
    K.NT_APPROXIMATE: ["clearance_constant"],
    K.NT_DESTEXHE: ["v_p", "k_p"],
    K.NT_DISCRETE_SPIKE: [],
    K.NT_EXPONENTIAL_DECAY: ["decay_constant"],
}
_RC_KIN_FIELDS = {
    K.RC_APPROXIMATE: ["r"],
    K.RC_DESTEXHE: ["r", "alpha", "beta"],
    K.RC_EXPONENTIAL_DECAY: ["r", "r_max", "decay_constant"],
}
_TYPE_NAMES = ["AMPA", "NMDA", "GABA"]


def _default_lattice_backend(model, ntk, rck, rows, cols):
    from .backend import CudaLatticeBackend
    return CudaLatticeBackend(model, ntk, rck, rows, cols)


def _default_network_backend(model, ntk, rck, train_kind, refract):
    from .backend import CudaNetworkBackend
    return CudaNetworkBackend(model, ntk, rck, train_kind, refract)


def _push_flag(owner, be, option, value, id=None):
    """Set an option that back ends without the feature need not know: only when it is on, or to switch it off again on the
    back end it was switched on for."""
    key = ("_flag_on", option)
    if value or owner.__dict__.get(key) is be:
        be.set_option(option, value, id)
    owner.__dict__[key] = be if value else None


def _enc(v):
    if v is None:
        return -1
    if isinstance(v, (bool, np.bool_)):
        return int(v)
    return v


class GridVoltageHistory:
    """neuron/mod.rs:286-301: `.history[step][row][col]`."""
    option = K.OPT_UPDATE_GRID_HISTORY

    def __init__(self, owner):
        self._o = owner

    @property
    def history(self):
        h = self._o._be.grid_history(self._o._bid)
        return h.reshape(h.shape[0], self._o.rows, self._o.cols)

    def reset(self):
        self._o._be.reset_history()


class SpikeHistory(GridVoltageHistory):
    """neuron/mod.rs:324-378: boolean raster; `aggregate()` = per-cell spike counts (:335-359)."""

    @property
    def history(self):
        h = self._o._be.spike_history(self._o._bid)
        return h.reshape(h.shape[0], self._o.rows, self._o.cols).astype(bool)

    def aggregate(self):
        """Per-cell spike counts over the recorded steps; the sum over steps is taken on the device (snn_*_get_spike_aggregate)."""
        return self._o._be.spike_aggregate(self._o._bid).reshape(self._o.rows, self._o.cols)


class SpikeEvents:
    """Spike events of one lattice (update_spike_events): record k holds the flat cell indices i*cols+j that spiked in the k-th
    recorded step, ascending, in `neurons[step_ptr[k]:step_ptr[k + 1]]`.  The same data as the dense SpikeHistory raster, without
    the steps x n grid: the compaction runs on the device and only the events reach the host."""

    def __init__(self, step_ptr, neurons, rows, cols):
        self.step_ptr = np.asarray(step_ptr, np.uint64)
        self.neurons = np.asarray(neurons, np.uint32)
        self.rows, self.cols = rows, cols

    @property
    def steps(self):
        return self.step_ptr.size - 1

    def _step_of_event(self):
        return np.repeat(np.arange(self.steps, dtype=np.int64), np.diff(self.step_ptr.astype(np.int64)))

    def pairs(self):
        """(n_events, 2) int64 array of (step, flat index): np.nonzero of the dense raster, in the same order."""
        return np.stack([self._step_of_event(), self.neurons.astype(np.int64)], axis=1)

    def dense(self):
        """The events expanded to the layout of spike_history.history: steps x rows x cols booleans."""
        out = np.zeros((self.steps, self.rows * self.cols), bool)
        out[self._step_of_event(), self.neurons.astype(np.int64)] = True
        return out.reshape(self.steps, self.rows, self.cols)


class AverageVoltageHistory(GridVoltageHistory):
    """neuron/mod.rs:303-322: `.history[step]` = mean membrane voltage of the lattice."""
    option = K.OPT_UPDATE_AVERAGE_HISTORY

    @property
    def history(self):
        return self._o._be.average_history(self._o._bid)


class EEGHistory(GridVoltageHistory):
    """neuron/mod.rs:231-284: `.history[step]` = (1 / (4 pi conductivity distance)) * sum(V - reference_voltage)."""
    option = K.OPT_UPDATE_EEG_HISTORY

    def __init__(self, owner, reference_voltage=0.007, distance=0.8, conductivity=251.0):
        super().__init__(owner)
        self.reference_voltage, self.distance, self.conductivity = reference_voltage, distance, conductivity

    @property
    def history(self):
        return self._o._be.eeg_history(self._o._bid)


class GraphHistory:
    """Graph::update_history (graph/mod.rs:278-284) of one graph: a lattice's own graph or one block of a network's connecting
    graph.  `.history[step]` holds every edge weight in the order of `row_ptr` / `pre` (CSR by postsynaptic cell, presynaptic
    cells ascending); `dense(step)` expands one record to the (connections, weights) layout of get_graph_dense.  A Lattice
    records after each step's plasticity, a LatticeNetwork before it (record 0 = the weights the first step read)."""

    def __init__(self, target):
        self._target = target   # () -> (back end, presynaptic id, postsynaptic id)

    @property
    def history(self):
        be, a, b = self._target()
        return be.graph_history(a, b)

    def _csr(self):
        be, a, b = self._target()
        return be.get_connection_csr(a, b)

    @property
    def row_ptr(self):
        return self._csr()[0]

    @property
    def pre(self):
        return self._csr()[1]

    def dense(self, step):
        be, a, b = self._target()
        rp, pre, _ = be.get_connection_csr(a, b)
        n_pre, n_post = be.size(a), be.size(b)
        post = np.repeat(np.arange(n_post), np.diff(rp.astype(np.int64)))
        conn, weights = np.zeros((n_pre, n_post), np.uint32), np.zeros((n_pre, n_post), np.float32)
        conn[pre, post] = 1
        weights[pre, post] = self.history[step]
        return conn, weights

    def reset(self):
        self._target()[0].reset_history()


class _CellLattice:
    """Shared by Lattice and SpikeTrainLattice: cell-grid <-> named SoA fields."""

    def __init__(self):
        self._be = None
        self._id = 0
        self._bid = 0   # id used on the back end: 0 for a stand-alone Lattice, the lattice id inside a network
        self.rows = 0
        self.cols = 0
        self.update_grid_history = False
        self.update_spike_history = False
        self.update_spike_events = False
        self.grid_history = GridVoltageHistory(self)
        self.spike_history = SpikeHistory(self)

    @property
    def spike_events(self):
        """The recorded spike events (SpikeEvents); cleared by spike_history.reset() / reset_history, not by reset_timing."""
        step_ptr, neurons = self._be.spike_events(self._bid)
        return SpikeEvents(step_ptr, neurons, self.rows, self.cols)

    # ---- field level (fast path) --------------------------------------------------------------
    @property
    def size(self):
        return self.rows * self.cols

    def get_field(self, name):
        return self._be.get_field(self._bid, name)

    def set_field(self, name, values):
        self._be.set_field(self._bid, name, values)

    def fill_field(self, name, value):
        self._be.fill_field(self._bid, name, _enc(value))

    def get_id(self):
        return self._id

    # ---- neurotransmitters of one cell <-> per-type arrays --------------------------------------
    def _rep(self, a):
        """Broadcast per-cell rows built for ONE base cell to the whole lattice (populate clones the base neuron)."""
        reps = getattr(self, "_uniform_reps", 1)
        return a if reps == 1 else np.tile(a, (reps,) + (1,) * (a.ndim - 1))

    def _upload_neurotransmitters(self, cells, ntk):
        n = len(cells)
        if not any(c.synaptic_neurotransmitters for c in cells):
            if not getattr(self, "_chem_touched", False):
                return
        self._chem_touched = True
        cls = NT_KINETICS[ntk]
        flags = np.zeros((n, 3), np.uint32)
        cols = {f: np.full((n, 3), cls._defaults[f], np.float32) for f in ["t", "t_max"] + _NT_PARAM_FIELDS[ntk]}
        for i, c in enumerate(cells):
            for ty, nt in c.synaptic_neurotransmitters.items():
                if nt.kind != ntk:
                    raise TypeError("all neurotransmitters of a lattice must use the same kinetics type")
                flags[i, int(ty)] = 1
                for f in cols:
                    cols[f][i, int(ty)] = getattr(nt, f)
        self.set_field("neurotransmitters$flags", self._rep(flags))
        for f, a in cols.items():
            self.set_field(f"neurotransmitters${f}", self._rep(a))

    def _download_neurotransmitters(self, cells, ntk):
        if not getattr(self, "_chem_touched", False):
            return
        n = len(cells)
        cls = NT_KINETICS[ntk]
        flags = self.get_field("neurotransmitters$flags").reshape(n, 3)
        cols = {f: self.get_field(f"neurotransmitters${f}").reshape(n, 3) for f in ["t", "t_max"] + _NT_PARAM_FIELDS[ntk]}
        for i, c in enumerate(cells):
            c.synaptic_neurotransmitters = {}
            for ty in range(3):
                if flags[i, ty]:
                    c.synaptic_neurotransmitters[IonotropicNeurotransmitterType(ty)] = cls(
                        **{f: float(cols[f][i, ty]) for f in cols})


class Lattice(_CellLattice):
    """Lattice<T, U, V, W, N> (neuron/mod.rs:556-587) with T = `neuron_type`, W = STDP."""

    def __init__(self, neuron_type=IzhikevichNeuron, id=0, backend_factory=None, history_type=GridVoltageHistory):
        """`history_type` mirrors the reference's LatticeHistory type parameter (GridVoltageHistory, AverageVoltageHistory
        or EEGHistory); `update_grid_history` switches whichever was chosen on."""
        super().__init__()
        self.grid_history = history_type(self)
        self.neuron_type = neuron_type
        self._id = id
        self._factory = backend_factory or _default_lattice_backend
        self._ntk = neuron_type.default_nt.kind
        self._rck = neuron_type.default_rc.kind
        # Lattice::default, neuron/mod.rs:589-606
        self.electrical_synapse = True
        self.chemical_synapse = False
        self.do_plasticity = False
        self.plasticity = STDP()
        self.parallel = False
        self.update_graph_history = False
        self.graph_history = GraphHistory(lambda: (self._be, self._bid, self._bid))
        self._in_network = None
        self._graph_spec = None  # remembered so that a lattice can be moved into a network

    @classmethod
    def default_impl(cls, neuron_type=IzhikevichNeuron, **kw):
        return cls(neuron_type, **kw)

    def set_id(self, id):
        if self._in_network is not None:
            raise RuntimeError("cannot change the id of a lattice inside a network")
        self._id = id

    # ---- populate / cell grid -----------------------------------------------------------------
    def _kinetics_of(self, neuron):
        ntk, rck = self._ntk, self._rck
        kinds = {nt.kind for nt in neuron.synaptic_neurotransmitters.values()}
        if len(kinds) > 1:
            raise TypeError("mixed neurotransmitter kinetics in one neuron")
        if kinds:
            ntk = kinds.pop()
        rk = {r.r.kind for r in neuron.receptors.values()}
        if len(rk) > 1:
            raise TypeError("mixed receptor kinetics in one neuron")
        if rk:
            rck = rk.pop()
        return ntk, rck

    def populate(self, base_neuron: Neuron, num_rows: int, num_cols: int):
        """neuron/mod.rs:1105-1126: clone the base neuron num_rows*num_cols times, nodes added row-major,
        any previous neurons and connections are dropped."""
        if self._in_network is not None:
            if (num_rows, num_cols) != (self.rows, self.cols):
                raise K.SnnError(K.SNN_GRAPH_DIMENSIONS_DO_NOT_MATCH, "Dimensions do not match")
        if not isinstance(base_neuron, self.neuron_type):
            raise TypeError(f"expected {self.neuron_type.__name__}")
        self._ntk, self._rck = self._kinetics_of(base_neuron)
        if self._in_network is None:
            if self._be is not None:
                self._be.close()
            self._be = self._factory(self.neuron_type.model, self._ntk, self._rck, num_rows, num_cols)
            self._bid = 0
        self.rows, self.cols = num_rows, num_cols
        self._graph_spec = None
        self._chem_touched = False
        if self.size == 0:
            return
        for name, v in base_neuron.scalar_fields().items():
            self.fill_field(name, v)
        if base_neuron.synaptic_neurotransmitters or base_neuron.receptors:
            # every cell is a clone of the base neuron: build the per-cell rows once and tile them (a Python loop over 10^8 cells
            # took minutes)
            self._uniform_reps = self.size
            try:
                self._upload_chem([base_neuron])
            finally:
                self._uniform_reps = 1

    def _upload_chem(self, cells):
        n = len(cells)
        self._upload_neurotransmitters(cells, self._ntk)
        if any(c.receptors for c in cells) or getattr(self, "_rc_touched", False):
            self._rc_touched = True
            flags = np.zeros((n, 3), np.uint32)
            arrs = {}
            for ty in range(3):
                rc_cls = RECEPTORS[IonotropicNeurotransmitterType(ty)]
                for f, d in rc_cls._defaults.items():
                    arrs[(ty, "_" + f)] = np.full(n, d, np.float32)
                for f in _RC_KIN_FIELDS[self._rck]:
                    arrs[(ty, "$r$kinetics$" + f)] = np.full(n, RC_KINETICS[self._rck]._defaults[f], np.float32)
            for i, c in enumerate(cells):
                for ty, rc in c.receptors.items():
                    ty = int(ty)
                    if int(rc.type) != ty:
                        # ReceptorNeurotransmitterError::MismatchedTypes (iterate_and_spike/mod.rs:1228-1254)
                        raise TypeError("Types are not compatible with one another")
                    if rc.r.kind != self._rck:
                        raise TypeError("all receptors of a lattice must use the same kinetics type")
                    flags[i, ty] = 1
                    for f in rc._defaults:
                        arrs[(ty, "_" + f)][i] = getattr(rc, f)
                    for f in _RC_KIN_FIELDS[self._rck]:
                        arrs[(ty, "$r$kinetics$" + f)][i] = getattr(rc.r, f)
            self.set_field("receptors$flags", self._rep(flags))
            for (ty, suffix), a in arrs.items():
                self.set_field(f"receptors${_TYPE_NAMES[ty]}{suffix}", self._rep(a))

    def cell_grid(self):
        """neuron/mod.rs:655-657 — materialised from the device fields."""
        n = self.size
        proto = self.neuron_type()
        cols = {name: self.get_field(name) for name in proto.scalar_fields()}
        cells = []
        for i in range(n):
            c = self.neuron_type()
            for name, a in cols.items():
                v = a[i]
                if name in ("is_spiking", "was_increasing"):
                    v = bool(v)
                elif name == "last_firing_time":
                    v = None if v < 0 else int(v)
                elif a.dtype.kind in "ui":   # usize fields (BCM period, num_spikes)
                    v = int(v)
                else:
                    v = float(v)
                c.scalar_fields()[name] = v
            cells.append(c)
        self._download_neurotransmitters(cells, self._ntk)
        if getattr(self, "_rc_touched", False):
            flags = self.get_field("receptors$flags").reshape(n, 3)
            for ty in range(3):
                if not flags[:, ty].any():
                    continue
                rc_cls = RECEPTORS[IonotropicNeurotransmitterType(ty)]
                fa = {f: self.get_field(f"receptors${_TYPE_NAMES[ty]}_{f}") for f in rc_cls._defaults}
                ka = {f: self.get_field(f"receptors${_TYPE_NAMES[ty]}$r$kinetics${f}") for f in _RC_KIN_FIELDS[self._rck]}
                for i in range(n):
                    if flags[i, ty]:
                        r = RC_KINETICS[self._rck](**{f: float(ka[f][i]) for f in ka})
                        cells[i].receptors[IonotropicNeurotransmitterType(ty)] = rc_cls(
                            r=r, **{f: float(fa[f][i]) for f in fa})
        return [cells[r * self.cols:(r + 1) * self.cols] for r in range(self.rows)]

    def set_cell_grid(self, cell_grid):
        """neuron/mod.rs:665-679: dimensions must match the existing grid."""
        if len(cell_grid) != self.rows or any(len(r) != self.cols for r in cell_grid):
            raise K.SnnError(K.SNN_GRAPH_POSITION_NOT_FOUND, "Position not found, position: Unmatched positions in new grid")
        cells = [c for row in cell_grid for c in row]
        if not cells:
            return
        for name in cells[0].scalar_fields():
            self.set_field(name, np.array([_enc(c.scalar_fields()[name]) for c in cells]))
        self._upload_chem(cells)

    def apply(self, f):
        """neuron/mod.rs:427-436."""
        grid = self.cell_grid()
        for row in grid:
            for neuron in row:
                f(neuron)
        self.set_cell_grid(grid)

    def apply_given_position(self, f):
        """neuron/mod.rs:440-449."""
        grid = self.cell_grid()
        for i, row in enumerate(grid):
            for j, neuron in enumerate(row):
                f((i, j), neuron)
        self.set_cell_grid(grid)

    # ---- graph --------------------------------------------------------------------------------
    def _positions(self):
        return [(i, j) for i in range(self.rows) for j in range(self.cols)]

    def connect(self, connecting_conditional, weight_logic=None):
        """neuron/mod.rs:1134-1157: every ordered pair of positions is evaluated; weight 1.0 when
        `weight_logic` is None; pairs failing the predicate become None."""
        pos = self._positions()
        n = len(pos)
        conn = np.zeros((n, n), np.uint32)
        w = np.zeros((n, n), np.float32)
        for a, x in enumerate(pos):
            for b, y in enumerate(pos):
                if connecting_conditional(x, y):
                    conn[a, b] = 1
                    w[a, b] = 1.0 if weight_logic is None else weight_logic(x, y)
        self._be.connect_dense(self._bid, self._bid, conn, w)
        self._graph_spec = ("dense", conn, w)

    def falliable_connect(self, connecting_conditional, weight_logic=None):
        """neuron/mod.rs:1165-1196 — predicate errors propagate to the caller."""
        self.connect(connecting_conditional, weight_logic)

    def connect_grid(self, radius=1, weight=1.0):
        """`connect(|x, y| max(|dr|,|dc|) <= radius && x != y, None)` built on the device."""
        self._be.connect_grid(self._bid, radius, weight)
        self._graph_spec = ("grid", radius, weight)

    def connect_csr(self, row_ptr, pre, weights):
        self._be.connect_csr(self._bid, self._bid, row_ptr, pre, weights)
        self._graph_spec = ("csr", np.array(row_ptr), np.array(pre), np.array(weights))

    def graph_dense(self):
        """(connections, weights) in the reference's GraphGPU layout [pre*n+post] (graph/mod.rs:300-361)."""
        return self._be.get_connection_dense(self._bid, self._bid)

    def graph_csr(self):
        return self._be.get_connection_csr(self._bid, self._bid)

    def get_weight(self, presynaptic, postsynaptic):
        """Graph::lookup_weight on (row, col) positions (graph/mod.rs:196-206); None = not connected."""
        for p, code in ((postsynaptic, K.SNN_GRAPH_POSTSYNAPTIC_NOT_FOUND), (presynaptic, K.SNN_GRAPH_PRESYNAPTIC_NOT_FOUND)):
            if not (0 <= p[0] < self.rows and 0 <= p[1] < self.cols):
                raise K.SnnError(code, f"position not found: {p}")
        a, b = presynaptic[0] * self.cols + presynaptic[1], postsynaptic[0] * self.cols + postsynaptic[1]
        if self._in_network is not None:
            return self._be.lookup_weight(self._bid, self._bid, a, b)
        return self._be.lookup_weight(a, b)

    def edit_weight(self, presynaptic, postsynaptic, weight):
        """Graph::edit_weight on (row, col) positions (graph/mod.rs:208-226); weight None removes the connection."""
        for p, code in ((postsynaptic, K.SNN_GRAPH_POSTSYNAPTIC_NOT_FOUND), (presynaptic, K.SNN_GRAPH_PRESYNAPTIC_NOT_FOUND)):
            if not (0 <= p[0] < self.rows and 0 <= p[1] < self.cols):
                raise K.SnnError(code, f"position not found: {p}")
        a, b = presynaptic[0] * self.cols + presynaptic[1], postsynaptic[0] * self.cols + postsynaptic[1]
        if self._in_network is not None:
            self._be.edit_weight(self._bid, self._bid, a, b, weight)
        else:
            self._be.edit_weight(a, b, weight)

    # ---- timing / options ---------------------------------------------------------------------
    @property
    def internal_clock(self):
        return self._be.get_option(K.OPT_INTERNAL_CLOCK)

    @internal_clock.setter
    def internal_clock(self, v):
        self._be.set_option(K.OPT_INTERNAL_CLOCK, v)

    def set_dt(self, dt):
        """neuron/mod.rs:649-652."""
        if self._in_network is not None:
            raise RuntimeError("use LatticeNetwork.set_dt for lattices inside a network")
        self._be.set_dt(dt)
        self.plasticity.dt = dt

    def reset_timing(self):
        """neuron/mod.rs:405-420."""
        self._be.reset_timing()

    def _push_options(self):
        be, i = self._be, self._bid
        if self._in_network is None:
            be.set_option(K.OPT_ELECTRICAL_SYNAPSE, self.electrical_synapse)
            be.set_option(K.OPT_CHEMICAL_SYNAPSE, self.chemical_synapse)
        be.set_option(K.OPT_DO_PLASTICITY, self.do_plasticity, i)
        gh = self.grid_history
        if isinstance(gh, EEGHistory):
            be.set_eeg_parameters(i, gh.reference_voltage, gh.distance, gh.conductivity)
        be.set_option(gh.option, self.update_grid_history, i)
        be.set_option(K.OPT_UPDATE_SPIKE_HISTORY, self.update_spike_history, i)
        _push_flag(self, be, K.OPT_UPDATE_SPIKE_EVENTS, self.update_spike_events, i)
        _push_flag(self, be, K.OPT_UPDATE_GRAPH_HISTORY, self.update_graph_history, i)
        p = self.plasticity
        if isinstance(p, BCM):   # Lattice<BCMIzhikevichNeuron, ..., BCM, ...>
            be.set_bcm_plasticity(i, True, p.decay, p.average_scalar, p.dt)
        else:
            if self.neuron_type.model == K.MODEL_BCM_IZH and self._in_network is None:
                be.set_bcm_plasticity(i, False, 0.1, 0.1, 0.1)
            be.set_plasticity(i, p.a_plus, p.a_minus, p.tau_plus, p.tau_minus, p.dt)

    def run_lattice(self, iterations: int):
        """RunLattice::run_lattice (neuron/mod.rs:1209-1219)."""
        if self._in_network is not None:
            raise RuntimeError("lattice is owned by a network; use run_lattices")
        if self._be is None:
            return  # never populated: empty lattice, Ok(()) (gpu_lattices/mod.rs:1089-1091)
        self._push_options()
        self._be.run(iterations)


class RewardModulatedLattice(Lattice):
    """RewardModulatedLattice<TraceRSTDP, T, ..., RewardModulatedSTDP, N> (neuron/mod.rs:2717-3416): same stepping as Lattice,
    but the graph holds TraceRSTDP weights and, while `do_modulation` is on, the reward modulator updates every edge twice per
    timestep (once from each end).  `run_lattice` steps without a reward signal (:3361-3374), `run_lattice_with_reward(r)` is
    one timestep preceded by `reward_modulator.update(r)` (:3250-3257); `run_lattice_with_rewards` batches such steps."""

    def __init__(self, neuron_type=IzhikevichNeuron, id=0, backend_factory=None, history_type=GridVoltageHistory):
        super().__init__(neuron_type, id, backend_factory, history_type)
        self.do_modulation = True                      # RewardModulatedLattice::default, neuron/mod.rs:2762-2777
        self.reward_modulator = RewardModulatedSTDP()

    def _push_options(self):
        self.do_plasticity = False
        super()._push_options()
        m = self.reward_modulator
        if self._in_network is not None:   # a member of RewardModulatedLatticeNetwork::reward_modulated_lattices
            self._be.set_lattice_reward_modulator(self._bid, self.do_modulation, **{k: getattr(m, k) for k in m._defaults})
        else:
            self._be.set_reward_modulator(True, self.do_modulation, **{k: getattr(m, k) for k in m._defaults})

    def _pull_modulator(self):
        if self._in_network is not None:
            self.reward_modulator.dopamine = self._be.get_lattice_reward_modulator(self._bid)[1]["dopamine"]
        else:
            self.reward_modulator.dopamine = self._be.get_reward_modulator()["dopamine"]

    def set_dt(self, dt):
        super().set_dt(dt)
        self.reward_modulator.dt = dt

    def run_lattice_with_reward(self, reward: float):
        self.run_lattice_with_rewards([reward])

    def run_lattice_with_rewards(self, rewards):
        if self._in_network is not None:
            raise RuntimeError("lattice is owned by a network; use run_lattices_with_reward")
        if self._be is None:
            return
        self._push_options()
        self._be.run_with_rewards(rewards)
        self._pull_modulator()

    def graph_traces(self):
        """(counter, dw, c) of every edge, in the order of graph_csr()."""
        self._push_options()
        if self._in_network is not None:
            return self._be.connection_traces(self._bid, self._bid)
        return self._be.connection_traces()

    def set_graph_traces(self, weight=None, counter=None, dw=None, c=None):
        """Graph::edit_weight with whole TraceRSTDP values on every existing edge (order of graph_csr(); None = keep)."""
        self._push_options()
        if self._in_network is not None:
            self._be.set_connection_traces(weight, counter, dw, c, pre_id=self._bid, post_id=self._bid)
        else:
            self._be.set_connection_traces(weight, counter, dw, c)


class SpikeTrainLattice(_CellLattice):
    """SpikeTrainLattice<N, T, U> (neuron/mod.rs:1290-1428)."""

    def __init__(self, spike_train_type=PoissonNeuron, id=0, network_backend_factory=None):
        super().__init__()
        self.spike_train_type = spike_train_type
        self._id = id
        self.id = id
        self._factory = network_backend_factory or _default_network_backend
        self._ntk = K.NT_APPROXIMATE
        self._refract = K.REFRACT_DELTA_DIRAC
        self._in_network = None
        self._cells_proto = None

    @classmethod
    def default_impl(cls, spike_train_type=PoissonNeuron, **kw):
        return cls(spike_train_type, **kw)

    def set_id(self, id):
        if self._in_network is not None:
            raise RuntimeError("cannot change the id of a lattice inside a network")
        self._id = self.id = id

    def populate(self, base_spike_train: SpikeTrain, num_rows: int, num_cols: int):
        """neuron/mod.rs:1397-1416."""
        if self._in_network is not None and (num_rows, num_cols) != (self.rows, self.cols):
            raise K.SnnError(K.SNN_GRAPH_DIMENSIONS_DO_NOT_MATCH, "Dimensions do not match")
        kinds = {nt.kind for nt in base_spike_train.synaptic_neurotransmitters.values()}
        if kinds:
            self._ntk = kinds.pop()
        self._refract = base_spike_train.neural_refractoriness.kind
        if self._in_network is None:
            if self._be is not None:
                self._be.close()
            # a stand-alone spike-train lattice is a network holding just this lattice
            self._be = self._factory(K.MODEL_IZH, self._ntk, K.RC_APPROXIMATE, self.spike_train_type.kind, self._refract)
            self._be.add_train_lattice(self._id, num_rows, num_cols)
            self._bid = self._id
        self.rows, self.cols = num_rows, num_cols
        self._chem_touched = False
        if self.size == 0:
            return
        self.set_spike_train_grid([[base_spike_train] * num_cols for _ in range(num_rows)])

    def set_spike_train_grid(self, grid):
        """neuron/mod.rs:1360-1374."""
        if len(grid) != self.rows or any(len(r) != self.cols for r in grid):
            raise K.SnnError(K.SNN_GRAPH_POSITION_NOT_FOUND, "Position not found, position: Unmatched positions in new grid")
        cells = [c for row in grid for c in row]
        if not cells:
            return
        for name in cells[0].scalar_fields():
            self.set_field(name, np.array([_enc(c.scalar_fields()[name]) for c in cells]))
        self.set_field("neural_refractoriness$k", np.array([c.neural_refractoriness.k for c in cells], np.float32))
        self._upload_neurotransmitters(cells, self._ntk)
        if self.spike_train_type.kind == K.TRAIN_PRESET:
            off = np.zeros(len(cells) + 1, np.uint64)
            off[1:] = np.cumsum([len(c.firing_times) for c in cells])
            times = np.array([t for c in cells for t in c.firing_times], np.float32)
            self._be.set_preset_firing_times(self._bid, off, times)
            self._firing_times = [list(c.firing_times) for c in cells]

    def spike_train_grid(self):
        n = self.size
        proto = self.spike_train_type()
        cols = {name: self.get_field(name) for name in proto.scalar_fields()}
        k = self.get_field("neural_refractoriness$k")
        cells = []
        for i in range(n):
            c = self.spike_train_type()
            for name, a in cols.items():
                v = a[i]
                if name == "is_spiking":
                    v = bool(v)
                elif name == "last_firing_time":
                    v = None if v < 0 else int(v)
                elif name == "counter":
                    v = int(v)
                else:
                    v = float(v)
                c.scalar_fields()[name] = v
            c.neural_refractoriness.k = float(k[i])
            if hasattr(self, "_firing_times"):
                c.firing_times = list(self._firing_times[i])
            cells.append(c)
        self._download_neurotransmitters(cells, self._ntk)
        return [cells[r * self.cols:(r + 1) * self.cols] for r in range(self.rows)]

    cell_grid = spike_train_grid

    def apply(self, f):
        grid = self.spike_train_grid()
        for row in grid:
            for s in row:
                f(s)
        self.set_spike_train_grid(grid)

    def apply_given_position(self, f):
        grid = self.spike_train_grid()
        for i, row in enumerate(grid):
            for j, s in enumerate(row):
                f((i, j), s)
        self.set_spike_train_grid(grid)

    @property
    def internal_clock(self):
        return self._be.get_option(K.OPT_INTERNAL_CLOCK, self._bid)

    @internal_clock.setter
    def internal_clock(self, v):
        self._be.set_option(K.OPT_INTERNAL_CLOCK, v, self._bid)

    def set_dt(self, dt):
        self._be.set_dt(dt)

    def reset_timing(self):
        self._be.reset_timing()

    def run_lattice(self, iterations: int):
        """RunSpikeTrainLattice::run_lattice (neuron/mod.rs:1419-1428)."""
        if self._in_network is not None:
            raise RuntimeError("lattice is owned by a network; use run_lattices")
        if self._be is None:
            return
        self._be.set_option(K.OPT_UPDATE_GRID_HISTORY, self.update_grid_history, self._bid)
        self._be.set_option(K.OPT_UPDATE_SPIKE_HISTORY, self.update_spike_history, self._bid)
        _push_flag(self, self._be, K.OPT_UPDATE_SPIKE_EVENTS, self.update_spike_events, self._bid)
        self._be.run(iterations)


class LatticeNetwork:
    """LatticeNetwork<...> (neuron/mod.rs:1538-1564)."""

    def __init__(self, backend_factory=None):
        self._factory = backend_factory or _default_network_backend
        self._be = None
        self._lattices = {}
        self._spike_train_lattices = {}
        # LatticeNetwork::default, neuron/mod.rs:1577-1588
        self.electrical_synapse = True
        self.chemical_synapse = False
        self.parallel = False
        self.update_connecting_graph_history = False

    @classmethod
    def default_impl(cls, **kw):
        return cls(**kw)

    def connecting_graph_history(self, presynaptic_id, postsynaptic_id):
        """Records of the connecting block presynaptic_id -> postsynaptic_id (update_connecting_graph_history)."""
        return GraphHistory(lambda: (self._be, presynaptic_id, postsynaptic_id))

    @classmethod
    def generate_network(cls, lattices, spike_train_lattices=(), backend_factory=None):
        """neuron/mod.rs:1625-1640."""
        net = cls(backend_factory)
        net._plan = (list(lattices), list(spike_train_lattices))
        model = lattices[0].neuron_type.model if lattices else K.MODEL_IZH
        ntk = lattices[0]._ntk if lattices else (spike_train_lattices[0]._ntk if spike_train_lattices else K.NT_APPROXIMATE)
        rck = lattices[0]._rck if lattices else K.RC_APPROXIMATE
        tk = spike_train_lattices[0].spike_train_type.kind if spike_train_lattices else K.TRAIN_POISSON
        rf = spike_train_lattices[0]._refract if spike_train_lattices else K.REFRACT_DELTA_DIRAC
        net._sig = (model, ntk, rck, tk, rf)
        net._be = net._factory(model, ntk, rck, tk, rf)
        for lat in lattices:
            net.add_lattice(lat)
        for st in spike_train_lattices:
            net.add_spike_train_lattice(st)
        return net

    def _ensure_backend(self, lat, train):
        if self._be is None:
            if train:
                sig = (K.MODEL_IZH, lat._ntk, K.RC_APPROXIMATE, lat.spike_train_type.kind, lat._refract)
            else:
                sig = (lat.neuron_type.model, lat._ntk, lat._rck, K.TRAIN_POISSON, K.REFRACT_DELTA_DIRAC)
            self._sig = sig
            self._be = self._factory(*sig)

    def get_all_ids(self):
        return set(self._lattices) | set(self._spike_train_lattices)

    def _adopt(self, lat, train):
        old_be, old_id = lat._be, lat._bid
        new_id = lat._id
        if old_be is not None and lat.size:
            names = list((lat.spike_train_type() if train else lat.neuron_type()).scalar_fields())
            if train:
                names.append("neural_refractoriness$k")
            if getattr(lat, "_chem_touched", False):
                cls_ = NT_KINETICS[lat._ntk]
                names += ["neurotransmitters$flags"] + [f"neurotransmitters${f}" for f in ["t", "t_max"] + _NT_PARAM_FIELDS[lat._ntk]]
                del cls_
            if getattr(lat, "_rc_touched", False):
                names.append("receptors$flags")
                for ty in range(3):
                    for f in RECEPTORS[IonotropicNeurotransmitterType(ty)]._defaults:
                        names.append(f"receptors${_TYPE_NAMES[ty]}_{f}")
                    for f in _RC_KIN_FIELDS[lat._rck]:
                        names.append(f"receptors${_TYPE_NAMES[ty]}$r$kinetics${f}")
            for name in names:
                self._be.set_field(new_id, name, old_be.get_field(old_id, name))
            if train and hasattr(lat, "_firing_times"):
                off = np.zeros(lat.size + 1, np.uint64)
                off[1:] = np.cumsum([len(t) for t in lat._firing_times])
                self._be.set_preset_firing_times(new_id, off, np.array([t for ts in lat._firing_times for t in ts], np.float32))
            if not train and lat._graph_spec is not None:
                rp, pr, w = old_be.get_connection_csr(old_id, old_id)
                self._be.connect_csr(new_id, new_id, rp, pr, w)
            clock = old_be.get_option(K.OPT_INTERNAL_CLOCK, old_id) if train else None
            if train and clock:
                self._be.set_option(K.OPT_INTERNAL_CLOCK, clock, new_id)
        if old_be is not None:
            old_be.close()
        lat._be, lat._in_network, lat._bid = self._be, self, new_id

    def add_lattice(self, lattice: Lattice):
        """neuron/mod.rs:1663-1678."""
        if lattice.get_id() in self.get_all_ids():
            raise K.SnnError(K.SNN_NET_GRAPH_ID_ALREADY_PRESENT, f"Graph id already present in network, id: {lattice.get_id()}")
        self._ensure_backend(lattice, False)
        if (lattice.neuron_type.model, lattice._rck) != (self._sig[0], self._sig[2]) and self._lattices:
            raise TypeError("all lattices of a network share one neuron / kinetics type")
        self._be.add_lattice(lattice.get_id(), lattice.rows, lattice.cols)
        self._adopt(lattice, False)
        self._lattices[lattice.get_id()] = lattice

    def add_spike_train_lattice(self, st: SpikeTrainLattice):
        """neuron/mod.rs:1682-1698."""
        if st.get_id() in self.get_all_ids():
            raise K.SnnError(K.SNN_NET_GRAPH_ID_ALREADY_PRESENT, f"Graph id already present in network, id: {st.get_id()}")
        self._ensure_backend(st, True)
        self._be.add_train_lattice(st.get_id(), st.rows, st.cols)
        self._adopt(st, True)
        self._spike_train_lattices[st.get_id()] = st

    def get_lattice(self, id):
        return self._lattices.get(id)

    def get_spike_train_lattice(self, id):
        return self._spike_train_lattices.get(id)

    def get_lattices(self):
        return self._lattices

    def get_spike_train_lattices(self):
        return self._spike_train_lattices

    def connect(self, presynaptic_id, postsynaptic_id, connecting_conditional, weight_logic=None):
        """neuron/mod.rs:1845-1930 (error order included)."""
        if postsynaptic_id in self._spike_train_lattices:
            raise K.SnnError(K.SNN_NET_POSTSYNAPTIC_LATTICE_CANNOT_BE_SPIKE_TRAIN,
                             "Postsynaptic lattice cannot be a spike train lattice because spike trains cannot take inputs")
        if presynaptic_id not in self.get_all_ids():
            raise K.SnnError(K.SNN_NET_PRESYNAPTIC_ID_NOT_FOUND, f"Presynaptic id not present in network, id: {presynaptic_id}")
        if postsynaptic_id not in self._lattices:
            raise K.SnnError(K.SNN_NET_POSTSYNAPTIC_ID_NOT_FOUND, f"Postsynaptic id not present in network, id: {postsynaptic_id}")
        if presynaptic_id == postsynaptic_id:
            return self.connect_interally(presynaptic_id, connecting_conditional, weight_logic)
        pre = self._lattices.get(presynaptic_id) or self._spike_train_lattices[presynaptic_id]
        post = self._lattices[postsynaptic_id]
        ppos = [(i, j) for i in range(pre.rows) for j in range(pre.cols)]
        qpos = post._positions()
        conn = np.zeros((len(ppos), len(qpos)), np.uint32)
        w = np.zeros((len(ppos), len(qpos)), np.float32)
        for a, x in enumerate(ppos):
            for b, y in enumerate(qpos):
                if connecting_conditional(x, y):
                    conn[a, b] = 1
                    w[a, b] = 1.0 if weight_logic is None else weight_logic(x, y)
        self._be.connect_dense(presynaptic_id, postsynaptic_id, conn, w)

    falliable_connect = connect

    def connect_interally(self, id, connecting_conditional, weight_logic=None):
        """neuron/mod.rs:2050-2063."""
        if id not in self._lattices:
            raise K.SnnError(K.SNN_NET_ID_NOT_FOUND_IN_LATTICES, f"Id not present in lattices, id: {id}")
        self._lattices[id].connect(connecting_conditional, weight_logic)

    def connection_dense(self, presynaptic_id, postsynaptic_id):
        return self._be.get_connection_dense(presynaptic_id, postsynaptic_id)

    @property
    def internal_clock(self):
        return self._be.get_option(K.OPT_INTERNAL_CLOCK)

    @internal_clock.setter
    def internal_clock(self, v):
        self._be.set_option(K.OPT_INTERNAL_CLOCK, v)

    def set_dt(self, dt):
        """neuron/mod.rs:1655-1660."""
        self._be.set_dt(dt)
        for lat in self._lattices.values():
            lat.plasticity.dt = dt

    def reset_timing(self):
        """neuron/mod.rs:1710-1717."""
        self._be.reset_timing()

    def run_lattices(self, iterations: int):
        """RunNetwork::run_lattices (neuron/mod.rs:2667-2674)."""
        if self._be is None:
            return
        self._be.set_option(K.OPT_ELECTRICAL_SYNAPSE, self.electrical_synapse)
        self._be.set_option(K.OPT_CHEMICAL_SYNAPSE, self.chemical_synapse)
        _push_flag(self, self._be, K.OPT_UPDATE_CONNECTING_GRAPH_HISTORY, self.update_connecting_graph_history)
        for lat in self._lattices.values():
            lat._push_options()
        for st in self._spike_train_lattices.values():
            self._be.set_option(K.OPT_UPDATE_GRID_HISTORY, st.update_grid_history, st.get_id())
            self._be.set_option(K.OPT_UPDATE_SPIKE_HISTORY, st.update_spike_history, st.get_id())
            _push_flag(st, self._be, K.OPT_UPDATE_SPIKE_EVENTS, st.update_spike_events, st.get_id())
        self._be.run(iterations)


class TraceRSTDP:
    """TraceRSTDP (plasticity/mod.rs:121-136): the weight type of reward-modulated graphs."""

    def __init__(self, counter=0, dw=0.0, weight=1.0, c=0.0):
        self.counter, self.dw, self.weight, self.c = counter, dw, weight, c

    def get_weight(self):
        return self.weight


class RewardModulatedConnection:
    """RewardModulatedConnection<S> (neuron/mod.rs:3418-3443): `Weight(f32)` or `RewardModulatedWeight(TraceRSTDP)`."""

    def __init__(self, value, reward_modulated):
        self.value, self.reward_modulated = value, reward_modulated

    @classmethod
    def Weight(cls, w):
        return cls(float(w), False)

    @classmethod
    def RewardModulatedWeight(cls, trace=None):
        return cls(trace if trace is not None else TraceRSTDP(), True)

    def get_weight(self):
        return self.value.weight if self.reward_modulated else self.value


class RewardModulatedLatticeNetwork(LatticeNetwork):
    """RewardModulatedLatticeNetwork<...> (neuron/mod.rs:3455-5455): plain lattices, reward-modulated lattices and spike-train
    lattices over one connecting graph of RewardModulatedConnection values.

    Differences from the reference, each refused with an error instead of silently diverging:
     * all edges of one connecting block (one presynaptic id -> postsynaptic id pair) hold the same connection kind;
     * the configurations on which the reference itself panics (connecting edges OUT of a reward-modulated lattice with
       do_modulation, or out of a plain lattice with do_plasticity: update_weights_from_neurons_across_*lattices looks them up
       with swapped end points, neuron/mod.rs:4760-4763, 4931-4934) make run_lattices raise SNN_UNSUPPORTED."""

    def __init__(self, backend_factory=None):
        super().__init__(backend_factory)
        self._reward_modulated_lattices = {}

    @classmethod
    def generate_network(cls, lattices, reward_modulated_lattices=(), spike_train_lattices=(), backend_factory=None):
        """neuron/mod.rs:3558-3594."""
        net = cls(backend_factory)
        neuron_lats = list(lattices) + list(reward_modulated_lattices)
        spike_train_lattices = list(spike_train_lattices)
        model = neuron_lats[0].neuron_type.model if neuron_lats else K.MODEL_IZH
        ntk = neuron_lats[0]._ntk if neuron_lats else (spike_train_lattices[0]._ntk if spike_train_lattices else K.NT_APPROXIMATE)
        rck = neuron_lats[0]._rck if neuron_lats else K.RC_APPROXIMATE
        tk = spike_train_lattices[0].spike_train_type.kind if spike_train_lattices else K.TRAIN_POISSON
        rf = spike_train_lattices[0]._refract if spike_train_lattices else K.REFRACT_DELTA_DIRAC
        net._sig = (model, ntk, rck, tk, rf)
        net._be = net._factory(model, ntk, rck, tk, rf)
        for lat in lattices:
            net.add_lattice(lat)
        for lat in reward_modulated_lattices:
            net.add_reward_modulated_lattice(lat)
        for st in spike_train_lattices:
            net.add_spike_train_lattice(st)
        return net

    def get_all_ids(self):
        return super().get_all_ids() | set(self._reward_modulated_lattices)

    def add_reward_modulated_lattice(self, lattice: RewardModulatedLattice):
        """neuron/mod.rs:3615-3634."""
        if lattice.get_id() in self.get_all_ids():
            raise K.SnnError(K.SNN_NET_GRAPH_ID_ALREADY_PRESENT, f"Graph id already present in network, id: {lattice.get_id()}")
        self._ensure_backend(lattice, False)
        if (lattice.neuron_type.model, lattice._rck) != (self._sig[0], self._sig[2]) and (self._lattices or self._reward_modulated_lattices):
            raise TypeError("all lattices of a network share one neuron / kinetics type")
        self._be.add_reward_lattice(lattice.get_id(), lattice.rows, lattice.cols)
        self._adopt(lattice, False)
        self._reward_modulated_lattices[lattice.get_id()] = lattice

    def get_reward_modulated_lattice(self, id):
        return self._reward_modulated_lattices.get(id)

    def get_reward_modulated_lattices(self):
        return self._reward_modulated_lattices

    def connect(self, presynaptic_id, postsynaptic_id, connecting_conditional, weight_logic=None):
        """neuron/mod.rs:3836-3947: plain / spike-train lattices only (error order included)."""
        if postsynaptic_id in self._spike_train_lattices:
            raise K.SnnError(K.SNN_NET_POSTSYNAPTIC_LATTICE_CANNOT_BE_SPIKE_TRAIN,
                             "Postsynaptic lattice cannot be a spike train lattice because spike trains cannot take inputs")
        if presynaptic_id not in self.get_all_ids():
            raise K.SnnError(K.SNN_NET_PRESYNAPTIC_ID_NOT_FOUND, f"Presynaptic id not present in network, id: {presynaptic_id}")
        msg = "Connect function must have non reward modulated lattices, connect with reward modulation instead"
        if postsynaptic_id not in self._lattices and postsynaptic_id in self._reward_modulated_lattices:
            raise K.SnnError(K.SNN_NET_CONNECT_FUNCTION_MUST_HAVE_NON_REWARD_MODULATED_LATTICE, msg)
        if postsynaptic_id in self._lattices and presynaptic_id in self._reward_modulated_lattices:
            raise K.SnnError(K.SNN_NET_CONNECT_FUNCTION_MUST_HAVE_NON_REWARD_MODULATED_LATTICE, msg)
        return super().connect(presynaptic_id, postsynaptic_id, connecting_conditional, weight_logic)

    falliable_connect = connect

    def connect_with_reward_modulation(self, presynaptic_id, postsynaptic_id, connecting_conditional, weight_logic):
        """neuron/mod.rs:4076-4209 (error order included).  `weight_logic(pre, post)` returns a RewardModulatedConnection."""
        if postsynaptic_id in self._spike_train_lattices:
            raise K.SnnError(K.SNN_NET_POSTSYNAPTIC_LATTICE_CANNOT_BE_SPIKE_TRAIN,
                             "Postsynaptic lattice cannot be a spike train lattice because spike trains cannot take inputs")
        if presynaptic_id not in self.get_all_ids():
            raise K.SnnError(K.SNN_NET_PRESYNAPTIC_ID_NOT_FOUND, f"Presynaptic id not present in network, id: {presynaptic_id}")
        rm = self._reward_modulated_lattices
        if postsynaptic_id not in rm and presynaptic_id not in rm:
            raise K.SnnError(K.SNN_NET_CANNOT_CONNECT_WITH_REWARD_MODULATED_CONNECTION,
                             "When connecting reward modulated network, at least one lattice has to be reward modulated")
        if postsynaptic_id not in self._lattices and postsynaptic_id not in rm:
            raise K.SnnError(K.SNN_NET_POSTSYNAPTIC_ID_NOT_FOUND, f"Postsynaptic id not present in network, id: {postsynaptic_id}")
        if presynaptic_id == postsynaptic_id:
            raise K.SnnError(K.SNN_NET_REWARD_MODULATED_CONNECTION_NOT_COMPATIBLE_INTERNALLY,
                             "When connecting reward modulated lattice, RewardModulatedConnection cannot be used to connect a "
                             "reward modulated lattice internally")
        pre = self._lattices.get(presynaptic_id) or rm.get(presynaptic_id) or self._spike_train_lattices[presynaptic_id]
        post = self._lattices.get(postsynaptic_id) or rm[postsynaptic_id]
        ppos = [(i, j) for i in range(pre.rows) for j in range(pre.cols)]
        qpos = post._positions()
        conn = np.zeros((len(ppos), len(qpos)), np.uint32)
        w = np.zeros((len(ppos), len(qpos)), np.float32)
        kinds, traces = set(), {}
        for a, x in enumerate(ppos):
            for b, y in enumerate(qpos):
                if connecting_conditional(x, y):
                    v = weight_logic(x, y)
                    conn[a, b] = 1
                    w[a, b] = v.get_weight()
                    kinds.add(v.reward_modulated)
                    if v.reward_modulated and (v.value.counter or v.value.dw or v.value.c):
                        traces[(a, b)] = v.value
        if len(kinds) > 1:
            raise K.SnnError(K.SNN_UNSUPPORTED, "one connecting block holds one kind of RewardModulatedConnection")
        self._be.connect_dense(presynaptic_id, postsynaptic_id, conn, w)
        if True in kinds:
            self._be.mark_connection_reward(presynaptic_id, postsynaptic_id, True)
            if traces:   # non-default TraceRSTDP members: written in the order of the block's CSR (post-major, pre ascending)
                order = [(a, b) for b in range(len(qpos)) for a in range(len(ppos)) if conn[a, b]]
                get = lambda k, f, d: getattr(traces[k], f) if k in traces else d
                self._be.set_connection_traces(None, [get(k, "counter", 0) for k in order], [get(k, "dw", 0.0) for k in order],
                                               [get(k, "c", 0.0) for k in order], pre_id=presynaptic_id, post_id=postsynaptic_id)

    falliable_connect_with_reward_modulation = connect_with_reward_modulation

    def connect_reward_modulated_lattice_interally(self, id, connecting_conditional, weight_logic=None):
        """neuron/mod.rs:4393-4413."""
        if id not in self._reward_modulated_lattices:
            raise K.SnnError(K.SNN_NET_ID_NOT_FOUND_IN_LATTICES, f"Id not present in lattices, id: {id}")
        self._reward_modulated_lattices[id].connect(connecting_conditional, weight_logic)

    def connection_traces(self, presynaptic_id, postsynaptic_id):
        """(counter, dw, c) of the block's edges in the order of its CSR (post-major, pre ascending)."""
        self._push_all()
        return self._be.connection_traces(presynaptic_id, postsynaptic_id)

    def set_dt(self, dt):
        """neuron/mod.rs:3666-3673."""
        super().set_dt(dt)
        for lat in self._reward_modulated_lattices.values():
            lat.plasticity.dt = dt
            lat.reward_modulator.dt = dt

    def _push_all(self):
        self._be.set_option(K.OPT_ELECTRICAL_SYNAPSE, self.electrical_synapse)
        self._be.set_option(K.OPT_CHEMICAL_SYNAPSE, self.chemical_synapse)
        _push_flag(self, self._be, K.OPT_UPDATE_CONNECTING_GRAPH_HISTORY, self.update_connecting_graph_history)
        for lat in list(self._lattices.values()) + list(self._reward_modulated_lattices.values()):
            lat._push_options()
        for st in self._spike_train_lattices.values():
            self._be.set_option(K.OPT_UPDATE_GRID_HISTORY, st.update_grid_history, st.get_id())
            self._be.set_option(K.OPT_UPDATE_SPIKE_HISTORY, st.update_spike_history, st.get_id())
            _push_flag(st, self._be, K.OPT_UPDATE_SPIKE_EVENTS, st.update_spike_events, st.get_id())

    def run_lattices(self, iterations: int):
        """RunNetwork::run_lattices (neuron/mod.rs:5411-5426): no reward signal."""
        if self._be is None:
            return
        self._push_all()
        self._be.run(iterations)

    def run_lattices_with_reward(self, reward: float):
        """neuron/mod.rs:5385-5392: one timestep, every modulator taking `reward` first."""
        self.run_lattices_with_rewards([reward])

    def run_lattices_with_rewards(self, rewards):
        if self._be is None:
            return
        self._push_all()
        self._be.run_network_with_rewards(rewards)
        for lat in self._reward_modulated_lattices.values():
            lat._pull_modulator()

    # Agent (neuron/mod.rs:5428-5455)
    def update_and_apply_reward(self, reward: float):
        self.run_lattices_with_reward(reward)

    def update(self):
        self.run_lattices(1)
