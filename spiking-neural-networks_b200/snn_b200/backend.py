"""CUDA back ends: thin object wrappers over the C ABI handles (snn_lattice_t / snn_network_t).

Both expose the same small protocol (methods take a lattice `id`; the single-lattice back end
ignores it) so the reference-shaped front end in lattice.py can drive either.  tests/ inject an
oracle back end with the same protocol; the product itself never imports the oracle.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi as K

_NP = {K.F32: np.float32, K.U32: np.uint32, K.I32: np.int32}


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _as(a, dtype) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=dtype)


class _CudaBase:
    network = False

    def __init__(self):
        self.lib = K.load_library()
        self.h = C.c_void_p()
        self._fields_cache = {}

    def _ck(self, status):
        K.check(self.lib, status, self.h, self.network)

    def close(self):
        if self.h:
            (self.lib.snn_network_destroy if self.network else self.lib.snn_lattice_destroy)(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- shared helpers -------------------------------------------------------------------------
    def fields(self, id=0):
        if id in self._fields_cache:
            return self._fields_cache[id]
        cnt = C.c_uint32()
        self._ck(self._field_count(id, C.byref(cnt)))
        out = []
        for i in range(cnt.value):
            name, dt, per = C.c_char_p(), C.c_int32(), C.c_uint32()
            self._ck(self._field_info(id, i, C.byref(name), C.byref(dt), C.byref(per)))
            out.append((name.value.decode(), dt.value, per.value))
        self._fields_cache[id] = out
        return out

    def field_meta(self, id, name):
        for n, dt, per in self.fields(id):
            if n == name:
                return dt, per
        raise K.SnnError(K.SNN_UNKNOWN_FIELD, f"unknown field: {name}")

    def set_field(self, id, name, arr):
        dt, _ = self.field_meta(id, name)
        a = _as(np.asarray(arr).reshape(-1), _NP[dt])
        self._ck(self._set_field(id, name.encode(), _ptr(a), a.size, dt))

    def get_field(self, id, name, out=None):
        """Read one named field.  `out` may be a preallocated (e.g. pinned) array of the right dtype and size."""
        dt, per = self.field_meta(id, name)
        if out is None:
            out = np.empty(self.size(id) * per, dtype=_NP[dt])
        elif out.dtype != _NP[dt] or out.size != self.size(id) * per or not out.flags.c_contiguous:
            raise ValueError(f"out buffer for {name} must be contiguous {_NP[dt].__name__}[{self.size(id) * per}]")
        self._ck(self._get_field(id, name.encode(), _ptr(out), out.size, dt))
        return out

    def fill_field(self, id, name, value):
        dt, _ = self.field_meta(id, name)
        fn = {K.F32: self._fill_f32, K.U32: self._fill_u32, K.I32: self._fill_i32}[dt]
        cast = {K.F32: float, K.U32: int, K.I32: int}[dt]
        self._ck(fn(id, name.encode(), cast(value)))

    def run(self, iterations):
        self._ck(self._run(int(iterations)))

    def run_timed(self, iterations):
        ms, nl = C.c_float(), C.c_uint64()
        self._ck(self._run_timed(int(iterations), C.byref(ms), C.byref(nl)))
        return ms.value, nl.value


class CudaLatticeBackend(_CudaBase):
    """snn_lattice_t: the LatticeGPU replacement (reference: gpu_lattices/mod.rs:327-511)."""

    def __init__(self, model, ntk=K.NT_APPROXIMATE, rck=K.RC_APPROXIMATE, rows=0, cols=0, device=-1, rank=0, world=1):
        super().__init__()
        d = K.LatticeDesc(C.sizeof(K.LatticeDesc), model, ntk, rck, rows, cols, device, rank, world)
        K.check(self.lib, self.lib.snn_lattice_create(C.byref(d), C.byref(self.h)))
        L = self.lib
        self._field_count = lambda id, p: L.snn_lattice_field_count(self.h, p)
        self._field_info = lambda id, i, a, b, c: L.snn_lattice_field_info(self.h, i, a, b, c)
        self._set_field = lambda id, n, p, c, d_: L.snn_lattice_set_field(self.h, n, p, c, d_)
        self._get_field = lambda id, n, p, c, d_: L.snn_lattice_get_field(self.h, n, p, c, d_)
        self._fill_f32 = lambda id, n, v: L.snn_lattice_fill_field_f32(self.h, n, v)
        self._fill_u32 = lambda id, n, v: L.snn_lattice_fill_field_u32(self.h, n, v)
        self._fill_i32 = lambda id, n, v: L.snn_lattice_fill_field_i32(self.h, n, v)
        self._run = lambda it: L.snn_lattice_run(self.h, it)
        self._run_timed = lambda it, a, b: L.snn_lattice_run_timed(self.h, it, a, b)

    def size(self, id=0):
        n = C.c_uint64()
        self._ck(self.lib.snn_lattice_size(self.h, C.byref(n)))
        return n.value

    def shape(self):
        r, c = C.c_uint32(), C.c_uint32()
        self._ck(self.lib.snn_lattice_rows(self.h, C.byref(r), C.byref(c)))
        return r.value, c.value

    def connect_dense(self, pre_id, post_id, connections, weights, index_to_position=None):
        c = _as(connections, np.uint32).reshape(-1)
        w = _as(weights, np.float32).reshape(-1)
        n = int(round(np.sqrt(c.size)))
        itp = None if index_to_position is None else _as(index_to_position, np.uint32)
        self._ck(self.lib.snn_lattice_set_graph_dense(self.h, _ptr(c), _ptr(w), None if itp is None else _ptr(itp), n))

    def connect_csr(self, pre_id, post_id, row_ptr, pre, weights):
        rp, pr, w = _as(row_ptr, np.uint64), _as(pre, np.uint32), _as(weights, np.float32)
        self._ck(self.lib.snn_lattice_set_graph_csr(self.h, _ptr(rp), _ptr(pr), _ptr(w), rp.size - 1, pr.size))

    def connect_grid(self, id, radius, weight):
        self._ck(self.lib.snn_lattice_set_graph_grid(self.h, int(radius), float(weight)))

    def connection_nnz(self, pre_id=0, post_id=0):
        n = C.c_uint64()
        self._ck(self.lib.snn_lattice_graph_nnz(self.h, C.byref(n)))
        return n.value

    def get_connection_csr(self, pre_id=0, post_id=0):
        n, nnz = self.size(), self.connection_nnz()
        rp = np.zeros(n + 1, np.uint64)
        pr = np.zeros(max(nnz, 1), np.uint32)
        w = np.zeros(max(nnz, 1), np.float32)
        self._ck(self.lib.snn_lattice_get_graph_csr(self.h, _ptr(rp), _ptr(pr), _ptr(w), n, nnz))
        return rp, pr[:nnz], w[:nnz]

    def get_connection_dense(self, pre_id=0, post_id=0):
        n = self.size()
        c = np.zeros(n * n, np.uint32)
        w = np.zeros(n * n, np.float32)
        self._ck(self.lib.snn_lattice_get_graph_dense(self.h, _ptr(c), _ptr(w), n))
        return c.reshape(n, n), w.reshape(n, n)

    def lookup_weight(self, pre, post):
        w, has = C.c_float(), C.c_int32()
        self._ck(self.lib.snn_lattice_lookup_weight(self.h, int(pre), int(post), C.byref(w), C.byref(has)))
        return w.value if has.value else None

    def edit_weight(self, pre, post, weight):
        """Graph::edit_weight(pre, post, Option<f32>): weight None removes the edge."""
        self._ck(self.lib.snn_lattice_edit_weight(self.h, int(pre), int(post), int(weight is not None),
                                                  0.0 if weight is None else float(weight)))

    def get_graph_rows(self, row_begin, row_end):
        """In-edges (CSR) of the postsynaptic positions [row_begin, row_end) with the current weights, read from the device table."""
        nrow = int(row_end) - int(row_begin)
        rp = np.zeros(nrow + 1, np.uint64)
        nnz = C.c_uint64()
        self._ck(self.lib.snn_lattice_get_graph_rows(self.h, int(row_begin), int(row_end), _ptr(rp), None, None, 0, C.byref(nnz)))
        pr, w = np.zeros(max(nnz.value, 1), np.uint32), np.zeros(max(nnz.value, 1), np.float32)
        self._ck(self.lib.snn_lattice_get_graph_rows(self.h, int(row_begin), int(row_end), _ptr(rp), _ptr(pr), _ptr(w), nnz.value, C.byref(nnz)))
        return rp, pr[:nnz.value], w[:nnz.value]

    def spike_aggregate(self, id=0):
        out = np.zeros(self.size(), np.int64)
        self._ck(self.lib.snn_lattice_get_spike_aggregate(self.h, _ptr(out), out.size))
        return out

    def set_option(self, option, value, id=None):
        self._ck(self.lib.snn_lattice_set_option(self.h, option, int(value)))

    def get_option(self, option, id=None):
        v = C.c_int64()
        self._ck(self.lib.snn_lattice_get_option(self.h, option, C.byref(v)))
        return v.value

    def set_plasticity(self, id, a_plus, a_minus, tau_plus, tau_minus, dt):
        s = K.StdpStruct(a_plus, a_minus, tau_plus, tau_minus, dt)
        self._ck(self.lib.snn_lattice_set_plasticity(self.h, C.byref(s)))

    _RSTDP = ("dopamine", "tau_d", "tau_c", "a_plus", "a_minus", "tau_plus", "tau_minus", "dt")

    def set_reward_modulator(self, enable, do_modulation, **m):
        """RewardModulatedLattice: the graph's weights become TraceRSTDP values updated by RewardModulatedSTDP."""
        s = K.RstdpStruct(*[float(m[k]) for k in self._RSTDP])
        self._ck(self.lib.snn_lattice_set_reward_modulator(self.h, int(enable), int(do_modulation), C.byref(s)))

    def get_reward_modulator(self):
        s = K.RstdpStruct()
        self._ck(self.lib.snn_lattice_get_reward_modulator(self.h, C.byref(s)))
        return {k: getattr(s, k) for k in self._RSTDP}

    def run_with_rewards(self, rewards):
        r = np.ascontiguousarray(np.asarray(rewards, np.float32).reshape(-1))
        self._ck(self.lib.snn_lattice_run_with_rewards(self.h, _ptr(r), r.size))

    def connection_traces(self):
        nnz = self.connection_nnz()
        cnt, dw, c = np.zeros(max(nnz, 1), np.uint32), np.zeros(max(nnz, 1), np.float32), np.zeros(max(nnz, 1), np.float32)
        self._ck(self.lib.snn_lattice_get_connection_traces(self.h, _ptr(cnt), _ptr(dw), _ptr(c), nnz))
        return cnt[:nnz], dw[:nnz], c[:nnz]

    def set_bcm_plasticity(self, id, enable, decay, average_scalar, dt):
        s = K.BcmStruct(decay, average_scalar, dt)
        self._ck(self.lib.snn_lattice_set_bcm_plasticity(self.h, int(enable), C.byref(s)))

    def set_connection_traces(self, weight=None, counter=None, dw=None, c=None):
        """Overwrite TraceRSTDP members of every edge in place (order of get_connection_csr; None = keep)."""
        nnz = self.connection_nnz()
        arrs = [None if x is None else _as(np.asarray(x).reshape(-1), t)
                for x, t in ((weight, np.float32), (counter, np.uint32), (dw, np.float32), (c, np.float32))]
        assert all(a is None or a.size == nnz for a in arrs)
        self._ck(self.lib.snn_lattice_set_connection_traces(self.h, *[None if a is None else _ptr(a) for a in arrs], nnz))

    def get_plasticity(self, id=0):
        s = K.StdpStruct()
        self._ck(self.lib.snn_lattice_get_plasticity(self.h, C.byref(s)))
        return s.a_plus, s.a_minus, s.tau_plus, s.tau_minus, s.dt

    def set_dt(self, dt):
        self._ck(self.lib.snn_lattice_set_dt(self.h, float(dt)))

    def reset_timing(self):
        self._ck(self.lib.snn_lattice_reset_timing(self.h))

    def history_len(self, id=0):
        n = C.c_uint64()
        self._ck(self.lib.snn_lattice_history_len(self.h, C.byref(n)))
        return n.value

    def grid_history(self, id=0):
        steps, n = self.history_len(), self.size()
        out = np.zeros(steps * n, np.float32)
        self._ck(self.lib.snn_lattice_get_grid_history(self.h, _ptr(out), out.size))
        return out.reshape(steps, n)

    def spike_history(self, id=0):
        steps, n = self.history_len(), self.size()
        out = np.zeros(steps * n, np.uint8)
        self._ck(self.lib.snn_lattice_get_spike_history(self.h, _ptr(out), out.size))
        return out.reshape(steps, n)

    def set_eeg_parameters(self, id, reference_voltage, distance, conductivity):
        self._ck(self.lib.snn_lattice_set_eeg_parameters(self.h, reference_voltage, distance, conductivity))

    def average_history(self, id=0):
        out = np.zeros(self.history_len(), np.float32)
        self._ck(self.lib.snn_lattice_get_average_history(self.h, _ptr(out), out.size))
        return out

    def eeg_history(self, id=0):
        out = np.zeros(self.history_len(), np.float32)
        self._ck(self.lib.snn_lattice_get_eeg_history(self.h, _ptr(out), out.size))
        return out

    def reset_history(self):
        self._ck(self.lib.snn_lattice_reset_history(self.h))

    def graph_history(self, pre_id=0, post_id=0):
        """Graph::update_history records of the lattice's graph: steps x nnz f32, edge order of get_connection_csr."""
        steps, nnz = C.c_uint64(), C.c_uint64()
        self._ck(self.lib.snn_lattice_graph_history_len(self.h, C.byref(steps), C.byref(nnz)))
        out = np.zeros(max(steps.value * nnz.value, 1), np.float32)
        self._ck(self.lib.snn_lattice_get_graph_history(self.h, _ptr(out), out.size))
        return out[:steps.value * nnz.value].reshape(steps.value, nnz.value)

    def spike_events(self, id=0):
        """Spike events of the lattice: (step_ptr u64[steps + 1], neurons u32[n_events]); record k is
        neurons[step_ptr[k]:step_ptr[k + 1]], global flat indices on a partitioned handle."""
        steps, n = C.c_uint64(), C.c_uint64()
        self._ck(self.lib.snn_lattice_spike_event_count(self.h, C.byref(steps), C.byref(n)))
        step_ptr, neurons = np.zeros(steps.value + 1, np.uint64), np.zeros(max(n.value, 1), np.uint32)
        self._ck(self.lib.snn_lattice_get_spike_events(self.h, _ptr(step_ptr), _ptr(neurons), neurons.size))
        return step_ptr, neurons[:n.value]

    # multi-GPU plumbing
    def ipc_export(self) -> bytes:
        buf = C.create_string_buffer(self.lib.snn_lattice_ipc_blob_size())
        self._ck(self.lib.snn_lattice_ipc_export(self.h, buf))
        return buf.raw

    def ipc_attach(self, direction: int, blob: bytes):
        buf = C.create_string_buffer(blob, len(blob))
        self._ck(self.lib.snn_lattice_ipc_attach(self.h, direction, buf))


    def attach_local(self, direction: int, neighbour: "CudaLatticeBackend"):
        """Attach a neighbouring strip that lives in this process (no CUDA IPC); call on both handles."""
        self._ck(self.lib.snn_lattice_attach_local(self.h, direction, neighbour.h))


    # general-graph partition (arbitrary in-edges across ranks)
    def gpart_wants(self, peer: int):
        """(ascending global indices of `peer`'s nodes this rank reads, first slot of them in this rank's node arrays)."""
        n, slot = C.c_uint64(), C.c_uint32()
        self._ck(self.lib.snn_lattice_gpart_wants(self.h, peer, None, 0, C.byref(n), C.byref(slot)))
        idx = np.zeros(max(n.value, 1), np.uint32)
        self._ck(self.lib.snn_lattice_gpart_wants(self.h, peer, _ptr(idx), idx.size, C.byref(n), C.byref(slot)))
        return idx[:n.value], slot.value

    def gpart_set_exports(self, peer: int, global_idx, first_slot_at_peer: int):
        idx = _as(global_idx, np.uint32)
        self._ck(self.lib.snn_lattice_gpart_set_exports(self.h, peer, _ptr(idx) if idx.size else None, idx.size, int(first_slot_at_peer)))

    def gpart_attach(self, peer: int, blob: bytes):
        buf = C.create_string_buffer(blob, len(blob))
        self._ck(self.lib.snn_lattice_gpart_attach(self.h, peer, buf))

    def gpart_attach_local(self, peer: int, other: "CudaLatticeBackend"):
        self._ck(self.lib.snn_lattice_gpart_attach_local(self.h, peer, other.h))


class CudaNetworkBackend(_CudaBase):
    """snn_network_t: the LatticeNetworkGPU replacement (reference: gpu_lattices/mod.rs:1560-1656)."""
    network = True

    def __init__(self, model, ntk=K.NT_APPROXIMATE, rck=K.RC_APPROXIMATE, train_kind=K.TRAIN_POISSON,
                 refract=K.REFRACT_DELTA_DIRAC, device=-1):
        super().__init__()
        d = K.NetworkDesc(C.sizeof(K.NetworkDesc), model, ntk, rck, train_kind, refract, device)
        K.check(self.lib, self.lib.snn_network_create(C.byref(d), C.byref(self.h)))
        L = self.lib
        self._field_count = lambda id, p: L.snn_network_field_count(self.h, id, p)
        self._field_info = lambda id, i, a, b, c: L.snn_network_field_info(self.h, id, i, a, b, c)
        self._set_field = lambda id, n, p, c, d_: L.snn_network_set_field(self.h, id, n, p, c, d_)
        self._get_field = lambda id, n, p, c, d_: L.snn_network_get_field(self.h, id, n, p, c, d_)
        self._fill_f32 = lambda id, n, v: L.snn_network_fill_field_f32(self.h, id, n, v)
        self._fill_u32 = lambda id, n, v: L.snn_network_fill_field_u32(self.h, id, n, v)
        self._fill_i32 = lambda id, n, v: L.snn_network_fill_field_i32(self.h, id, n, v)
        self._run = lambda it: L.snn_network_run(self.h, it)
        self._run_timed = lambda it, a, b: L.snn_network_run_timed(self.h, it, a, b)

    def add_lattice(self, id, rows, cols):
        self._ck(self.lib.snn_network_add_lattice(self.h, id, rows, cols))

    def add_train_lattice(self, id, rows, cols):
        self._ck(self.lib.snn_network_add_spike_train_lattice(self.h, id, rows, cols))

    # ---- RewardModulatedLatticeNetwork (neuron/mod.rs:3455-5455) ----
    _RSTDP = ("dopamine", "tau_d", "tau_c", "a_plus", "a_minus", "tau_plus", "tau_minus", "dt")

    def add_reward_lattice(self, id, rows, cols):
        self._ck(self.lib.snn_network_add_reward_modulated_lattice(self.h, id, rows, cols))

    def set_lattice_reward_modulator(self, id, do_modulation, **m):
        s = K.RstdpStruct(*[float(m[k]) for k in self._RSTDP])
        self._ck(self.lib.snn_network_set_reward_modulator(self.h, id, int(do_modulation), C.byref(s)))

    def get_lattice_reward_modulator(self, id):
        s, dm = K.RstdpStruct(), C.c_int32(0)
        self._ck(self.lib.snn_network_get_reward_modulator(self.h, id, C.byref(dm), C.byref(s)))
        return bool(dm.value), {k: getattr(s, k) for k in self._RSTDP}

    def mark_connection_reward(self, pre_id, post_id, reward_modulated):
        self._ck(self.lib.snn_network_set_connection_reward_modulated(self.h, pre_id, post_id, int(reward_modulated)))

    def run_network_with_rewards(self, rewards):
        r = np.ascontiguousarray(np.asarray(rewards, np.float32).reshape(-1))
        self._ck(self.lib.snn_network_run_with_rewards(self.h, _ptr(r), r.size))

    def connection_traces(self, pre_id, post_id):
        nnz = self.connection_nnz(pre_id, post_id)
        cnt, dw, c = np.zeros(max(nnz, 1), np.uint32), np.zeros(max(nnz, 1), np.float32), np.zeros(max(nnz, 1), np.float32)
        self._ck(self.lib.snn_network_get_connection_traces(self.h, pre_id, post_id, _ptr(cnt), _ptr(dw), _ptr(c), nnz))
        return cnt[:nnz], dw[:nnz], c[:nnz]

    def set_connection_traces(self, weight=None, counter=None, dw=None, c=None, pre_id=0, post_id=0):
        nnz = self.connection_nnz(pre_id, post_id)
        arrs = [None if x is None else _as(np.asarray(x).reshape(-1), t)
                for x, t in ((weight, np.float32), (counter, np.uint32), (dw, np.float32), (c, np.float32))]
        self._ck(self.lib.snn_network_set_connection_traces(self.h, pre_id, post_id, *[None if a is None else _ptr(a) for a in arrs], nnz))

    def size(self, id):
        n = C.c_uint64()
        self._ck(self.lib.snn_network_lattice_size(self.h, id, C.byref(n)))
        return n.value

    def set_preset_firing_times(self, id, offsets, times):
        off, t = _as(offsets, np.uint64), _as(times, np.float32)
        self._ck(self.lib.snn_network_set_preset_firing_times(self.h, id, _ptr(off), _ptr(t), off.size - 1, t.size))

    def connect_dense(self, pre_id, post_id, connections, weights, index_to_position=None):
        c = _as(connections, np.uint32)
        w = _as(weights, np.float32)
        n_pre, n_post = self.size(pre_id), self.size(post_id)
        self._ck(self.lib.snn_network_connect_dense(self.h, pre_id, post_id, _ptr(c), _ptr(w), n_pre, n_post))

    def connect_csr(self, pre_id, post_id, row_ptr, pre, weights):
        rp, pr, w = _as(row_ptr, np.uint64), _as(pre, np.uint32), _as(weights, np.float32)
        self._ck(self.lib.snn_network_connect_csr(self.h, pre_id, post_id, _ptr(rp), _ptr(pr), _ptr(w), rp.size - 1, pr.size))

    def connection_nnz(self, pre_id, post_id):
        n = C.c_uint64()
        self._ck(self.lib.snn_network_connection_nnz(self.h, pre_id, post_id, C.byref(n)))
        return n.value

    def get_connection_csr(self, pre_id, post_id):
        n, nnz = self.size(post_id), self.connection_nnz(pre_id, post_id)
        rp = np.zeros(n + 1, np.uint64)
        pr = np.zeros(max(nnz, 1), np.uint32)
        w = np.zeros(max(nnz, 1), np.float32)
        self._ck(self.lib.snn_network_get_connection_csr(self.h, pre_id, post_id, _ptr(rp), _ptr(pr), _ptr(w), n, nnz))
        return rp, pr[:nnz], w[:nnz]

    def get_connection_dense(self, pre_id, post_id):
        n_pre, n_post = self.size(pre_id), self.size(post_id)
        c = np.zeros(n_pre * n_post, np.uint32)
        w = np.zeros(n_pre * n_post, np.float32)
        self._ck(self.lib.snn_network_get_connection_dense(self.h, pre_id, post_id, _ptr(c), _ptr(w), n_pre, n_post))
        return c.reshape(n_pre, n_post), w.reshape(n_pre, n_post)

    def lookup_weight(self, pre_id, post_id, pre, post):
        w, has = C.c_float(), C.c_int32()
        self._ck(self.lib.snn_network_lookup_weight(self.h, pre_id, post_id, int(pre), int(post), C.byref(w), C.byref(has)))
        return w.value if has.value else None

    def edit_weight(self, pre_id, post_id, pre, post, weight):
        self._ck(self.lib.snn_network_edit_weight(self.h, pre_id, post_id, int(pre), int(post), int(weight is not None),
                                                  0.0 if weight is None else float(weight)))

    def spike_aggregate(self, id):
        out = np.zeros(self.size(id), np.int64)
        self._ck(self.lib.snn_network_get_spike_aggregate(self.h, id, _ptr(out), out.size))
        return out

    def set_option(self, option, value, id=None):
        if id is None:
            self._ck(self.lib.snn_network_set_option(self.h, option, int(value)))
        else:
            self._ck(self.lib.snn_network_set_lattice_option(self.h, id, option, int(value)))

    def get_option(self, option, id=None):
        v = C.c_int64()
        if id is None:
            self._ck(self.lib.snn_network_get_option(self.h, option, C.byref(v)))
        else:
            self._ck(self.lib.snn_network_get_lattice_option(self.h, id, option, C.byref(v)))
        return v.value

    def set_plasticity(self, id, a_plus, a_minus, tau_plus, tau_minus, dt):
        s = K.StdpStruct(a_plus, a_minus, tau_plus, tau_minus, dt)
        self._ck(self.lib.snn_network_set_plasticity(self.h, id, C.byref(s)))

    def set_dt(self, dt):
        self._ck(self.lib.snn_network_set_dt(self.h, float(dt)))

    def reset_timing(self):
        self._ck(self.lib.snn_network_reset_timing(self.h))

    def history_len(self, id):
        n = C.c_uint64()
        self._ck(self.lib.snn_network_history_len(self.h, id, C.byref(n)))
        return n.value

    def grid_history(self, id):
        steps, n = self.history_len(id), self.size(id)
        out = np.zeros(steps * n, np.float32)
        self._ck(self.lib.snn_network_get_grid_history(self.h, id, _ptr(out), out.size))
        return out.reshape(steps, n)

    def spike_history(self, id):
        steps, n = self.history_len(id), self.size(id)
        out = np.zeros(steps * n, np.uint8)
        self._ck(self.lib.snn_network_get_spike_history(self.h, id, _ptr(out), out.size))
        return out.reshape(steps, n)

    def set_eeg_parameters(self, id, reference_voltage, distance, conductivity):
        self._ck(self.lib.snn_network_set_eeg_parameters(self.h, id, reference_voltage, distance, conductivity))

    def average_history(self, id):
        out = np.zeros(self.history_len(id), np.float32)
        self._ck(self.lib.snn_network_get_average_history(self.h, id, _ptr(out), out.size))
        return out

    def eeg_history(self, id):
        out = np.zeros(self.history_len(id), np.float32)
        self._ck(self.lib.snn_network_get_eeg_history(self.h, id, _ptr(out), out.size))
        return out

    def reset_history(self):
        self._ck(self.lib.snn_network_reset_history(self.h))

    def graph_history(self, pre_id, post_id):
        """Records of the block pre_id -> post_id (a lattice's own graph when equal): steps x nnz f32, edge order of
        get_connection_csr(pre_id, post_id)."""
        steps, nnz = C.c_uint64(), C.c_uint64()
        self._ck(self.lib.snn_network_graph_history_len(self.h, pre_id, post_id, C.byref(steps), C.byref(nnz)))
        out = np.zeros(max(steps.value * nnz.value, 1), np.float32)
        self._ck(self.lib.snn_network_get_graph_history(self.h, pre_id, post_id, _ptr(out), out.size))
        return out[:steps.value * nnz.value].reshape(steps.value, nnz.value)

    def spike_events(self, id):
        """Spike events of lattice `id`: (step_ptr u64[steps + 1], neurons u32[n_events]), indices inside the lattice."""
        steps, n = C.c_uint64(), C.c_uint64()
        self._ck(self.lib.snn_network_spike_event_count(self.h, id, C.byref(steps), C.byref(n)))
        step_ptr, neurons = np.zeros(steps.value + 1, np.uint64), np.zeros(max(n.value, 1), np.uint32)
        self._ck(self.lib.snn_network_get_spike_events(self.h, id, _ptr(step_ptr), _ptr(neurons), neurons.size))
        return step_ptr, neurons[:n.value]
