"""Graph::update_history (graph/mod.rs:278-284) on top of the CPU oracle, for tests/test_graph_history.py.

The oracle library itself records no graph history; this back end steps it one timestep at a time and copies every recorded
graph literally, at the placement the reference uses for each handle kind:
  * a Lattice (the lattice-role back end, created with rows / cols) pushes its graph history at the end of Lattice::iterate, after
    the step's plasticity (neuron/mod.rs:973-979): the weights read after the step;
  * a LatticeNetwork pushes each lattice's graph history and the connecting-graph history before the step's STDP
    (neuron/mod.rs:2565-2576): the weights read before the step.
It also enforces the product's rules: no adjacency change while records exist, no records for reward-modulated lattices.
"""
from __future__ import annotations

import numpy as np

from oracle_api import OracleBackend, OracleError
from snn_b200 import _capi as K


class GraphHistoryOracle(OracleBackend):
    def __init__(self, model, ntk=0, rck=0, train_kind=0, refract=0, rows=None, cols=None):
        self._lattice_role = rows is not None
        self._neuron_ids, self._train_ids = [], []
        self._reward = False
        self._gh_lattices, self._gh_connecting = set(), False
        self._records = {}
        super().__init__(model, ntk, rck, train_kind, refract, rows=rows, cols=cols)

    # ---- lattices -------------------------------------------------------------------------------
    def add_lattice(self, id, rows, cols):
        super().add_lattice(id, rows, cols)
        self._neuron_ids.append(id)

    def add_reward_lattice(self, id, rows, cols):
        super().add_reward_lattice(id, rows, cols)
        self._neuron_ids.append(id)
        self._reward = True

    def add_train_lattice(self, id, rows, cols):
        super().add_train_lattice(id, rows, cols)
        self._train_ids.append(id)

    def set_reward_modulator(self, enable, do_modulation, **m):
        super().set_reward_modulator(enable, do_modulation, **m)
        self._reward = bool(enable)

    # ---- options --------------------------------------------------------------------------------
    def set_option(self, option, value, id=None):
        if option == K.OPT_UPDATE_GRAPH_HISTORY:
            (self._gh_lattices.add if value else self._gh_lattices.discard)(0 if id is None else id)
        elif option == K.OPT_UPDATE_CONNECTING_GRAPH_HISTORY:
            self._gh_connecting = bool(value)
        else:
            super().set_option(option, value, id)

    # ---- adjacency is frozen while records exist --------------------------------------------------
    def _recording_started(self):
        return any(len(v) for v in self._records.values())

    def connect_dense(self, *a, **kw):
        if self._recording_started():
            raise OracleError(K.SNN_UNSUPPORTED)
        super().connect_dense(*a, **kw)

    def connect_grid(self, *a, **kw):
        if self._recording_started():
            raise OracleError(K.SNN_UNSUPPORTED)
        super().connect_grid(*a, **kw)

    def connect_csr(self, pre_id, post_id, row_ptr, pre, weights):
        # OracleBackend.edit_weight rewrites the block through here: a weight-only edit keeps the adjacency and is allowed
        if self._recording_started():
            rp, pr, _ = self.get_connection_csr(pre_id, post_id)
            rp2, pr2 = np.asarray(row_ptr, np.uint64), np.asarray(pre, np.uint32)
            if rp.shape != rp2.shape or (rp != rp2).any() or pr.shape != pr2.shape or (pr != pr2).any():
                raise OracleError(K.SNN_UNSUPPORTED)
        super().connect_csr(pre_id, post_id, row_ptr, pre, weights)

    # ---- recording ------------------------------------------------------------------------------
    def _keys(self):
        keys = [(i, i) for i in self._neuron_ids if i in self._gh_lattices]
        if self._gh_connecting:
            keys += [(a, b) for b in self._neuron_ids for a in self._neuron_ids + self._train_ids
                     if a != b and self.connection_nnz(a, b)]
        return keys

    def _push(self, keys):
        for k in keys:
            self._records.setdefault(k, []).append(self.get_connection_csr(*k)[2].copy())

    def run(self, iterations):
        keys = self._keys()
        if not keys:
            return super().run(iterations)
        if self._reward:
            raise OracleError(K.SNN_UNSUPPORTED)   # TraceRSTDP records are not defined
        if not getattr(self, "_el", 1) and not getattr(self, "_ch", 0):
            return super().run(iterations)        # run_lattice with both synapse kinds off is a no-op
        for _ in range(int(iterations)):
            if not self._lattice_role:
                self._push(keys)
            super().run(1)
            if self._lattice_role:
                self._push(keys)

    def run_with_rewards(self, rewards):
        if self._keys():
            raise OracleError(K.SNN_UNSUPPORTED)
        super().run_with_rewards(rewards)

    def run_network_with_rewards(self, rewards):
        if self._keys():
            raise OracleError(K.SNN_UNSUPPORTED)
        super().run_network_with_rewards(rewards)

    def graph_history(self, pre_id=0, post_id=0):
        rec = self._records.get((pre_id, post_id))
        if not rec:
            return np.zeros((0, 0), np.float32)
        return np.array(rec, np.float32).reshape(len(rec), -1)

    def reset_history(self):
        super().reset_history()
        self._records = {}
