"""Multi-GPU row-strip lattices: one process per GPU, torch.distributed only for plumbing.

The data path has no host-driven collective: each rank's fused step kernel pushes its boundary rows
(V, last_firing_time, neurotransmitter t) straight into the neighbouring GPUs' ghost slots over NVLink
peer memory and raises an arrival counter there; the neighbour's boundary warps spin on that counter
before they gather (csrc/kernels.cu).  torch.distributed moves the CUDA-IPC blobs once at set-up and
provides barriers around timing.
"""
from __future__ import annotations

from . import _capi as K
from .backend import CudaLatticeBackend
from .lattice import SpikeEvents


def partition_rows(rows: int, world: int, rank: int):
    """[begin, end) of `rank`'s strip — the library's own host-side plan (snn_partition_begin)."""
    lib = K.load_library()
    return lib.snn_partition_begin(rows, world, rank), lib.snn_partition_begin(rows, world, rank + 1)


def exchange_blobs(blob: bytes, rank: int, world: int, group=None):
    """all-gather of the opaque IPC blobs; returns (blob of rank-1 or None, blob of rank+1 or None)."""
    import torch.distributed as dist
    blobs = [None] * world
    dist.all_gather_object(blobs, blob, group=group)
    return (blobs[rank - 1] if rank > 0 else None), (blobs[rank + 1] if rank < world - 1 else None)


def merge_spike_events(parts, rows, cols):
    """One SpikeEvents of the whole lattice from every rank's (step_ptr, neurons), in rank order: record k is the ranks' records k
    one after the other.  Ranks own contiguous rows in rank order, so that is already ascending global order."""
    import numpy as np
    steps = {p[0].size - 1 for p in parts}
    if len(steps) != 1:
        raise ValueError(f"the ranks hold different numbers of spike-event records: {sorted(steps)}")
    steps = steps.pop()
    counts = np.stack([np.diff(p[0].astype(np.int64)) for p in parts])   # ranks x steps
    step_ptr = np.zeros(steps + 1, np.uint64)
    step_ptr[1:] = np.cumsum(counts.sum(axis=0))
    step_of = np.concatenate([np.repeat(np.arange(steps), c) for c in counts]) if steps else np.zeros(0, np.int64)
    neurons = np.concatenate([p[1] for p in parts]) if parts else np.zeros(0, np.uint32)
    order = np.argsort(step_of, kind="stable")   # stable: the ranks stay in rank order inside a step
    return SpikeEvents(step_ptr, neurons[order], rows, cols)


def gather_spike_events(be, rank, world, group=None):
    """torch.distributed: every rank's spike events of a row-strip or general-graph partition, merged as merge_spike_events does
    (one all_gather_object); returns the whole lattice's SpikeEvents on every rank."""
    import torch.distributed as dist
    parts = [None] * world
    dist.all_gather_object(parts, (be.spike_events(), be.shape()), group=group)
    rows, cols = sum(p[1][0] for p in parts), parts[0][1][1]
    return merge_spike_events([p[0] for p in parts], rows, cols)


class StripLattice:
    """A lattice of `rows` x `cols` neurons split into contiguous row strips, one per rank."""

    def __init__(self, model, rows, cols, rank, world, ntk=K.NT_APPROXIMATE, rck=K.RC_APPROXIMATE, device=-1):
        self.rank, self.world = rank, world
        self.rows, self.cols = rows, cols
        self.row_begin, self.row_end = partition_rows(rows, world, rank)
        self.be = CudaLatticeBackend(model, ntk, rck, rows, cols, device=device, rank=rank, world=world)
        self.local_rows = self.row_end - self.row_begin
        self.n_local = self.local_rows * cols

    def attach(self, group=None):
        """Export my halo-visible slab, gather everyone's, map the two neighbours.  Call after the fields that
        decide the memory layout (chemistry on/off, stencil radius) have been set."""
        if self.world == 1:
            return
        import torch.distributed as dist
        lo, hi = exchange_blobs(self.be.ipc_export(), self.rank, self.world, group)
        if lo is not None:
            self.be.ipc_attach(-1, lo)
        if hi is not None:
            self.be.ipc_attach(+1, hi)
        dist.barrier(group=group)


def attach_general(be, rank, world, group=None):
    """General-graph partition set-up for this rank (after snn_lattice_set_graph_csr with global indices on every rank): exchange
    the gather lists and the IPC blobs, map every peer this rank exchanges with.  One all_gather_object of small host objects."""
    import torch.distributed as dist
    wants = {q: be.gpart_wants(q) for q in range(world) if q != rank}
    mine = {"wants": {q: (idx, slot) for q, (idx, slot) in wants.items() if idx.size}, "blob": None}
    everyone = [None] * world
    dist.all_gather_object(everyone, mine, group=group)
    peers = set(mine["wants"].keys())
    for q in range(world):
        if q != rank and rank in everyone[q]["wants"]:
            idx, slot = everyone[q]["wants"][rank]
            be.gpart_set_exports(q, idx, slot)
            peers.add(q)
    blobs = [None] * world
    dist.all_gather_object(blobs, be.ipc_export() if peers else None, group=group)
    for q in sorted(peers):
        be.gpart_attach(q, blobs[q])
    dist.barrier(group=group)
    return sorted(peers)


class LocalStrips:
    """The same row-strip partition with every strip in THIS process (snn_lattice_attach_local): strips on one device, or one
    process driving several GPUs.  `run` steps all strips concurrently from one host thread each (a strip's boundary warps wait
    for its neighbours' progress on the device, so the calls must overlap).  On a single device the strips' kernels must be able
    to run concurrently: keep them small, and raise CUDA_DEVICE_MAX_CONNECTIONS (before CUDA starts) so that no two of the
    handles' streams share a hardware work queue."""

    def __init__(self, model, rows, cols, world, ntk=K.NT_APPROXIMATE, rck=K.RC_APPROXIMATE, devices=None):
        self.rows, self.cols, self.world = rows, cols, world
        self.bounds = [partition_rows(rows, world, r)[0] for r in range(world)] + [rows]
        devices = devices or [-1] * world
        self.strips = [CudaLatticeBackend(model, ntk, rck, rows, cols, device=devices[r], rank=r, world=world) for r in range(world)]

    def rows_of(self, r):
        return slice(self.bounds[r] * self.cols, self.bounds[r + 1] * self.cols)

    def set_field(self, name, arr, per=1):
        import numpy as np
        a = np.asarray(arr).reshape(self.rows * self.cols, per)
        for r, be in enumerate(self.strips):
            be.set_field(0, name, a[self.rows_of(r)].reshape(-1))

    def get_field(self, name):
        import numpy as np
        return np.concatenate([be.get_field(0, name) for be in self.strips])

    def each(self, fn):
        for be in self.strips:
            fn(be)

    def attach(self):
        for r, be in enumerate(self.strips):
            if r > 0:
                be.attach_local(-1, self.strips[r - 1])
            if r < self.world - 1:
                be.attach_local(+1, self.strips[r + 1])

    def set_graph_csr(self, row_ptr, pre, weights):
        """Whole-lattice CSR (global indices) cut into the strips' rows; edges may reach any node (general-graph partition)."""
        import numpy as np
        rp, pre, w = np.asarray(row_ptr, np.uint64), np.asarray(pre, np.uint32), np.asarray(weights, np.float32)
        for r, be in enumerate(self.strips):
            be.set_option(K.OPT_GENERAL_PARTITION, 1)   # the same mode on every rank
            q0, q1 = self.bounds[r] * self.cols, self.bounds[r + 1] * self.cols
            s, t = int(rp[q0]), int(rp[q1])
            be.connect_csr(0, 0, rp[q0:q1 + 1] - rp[q0], pre[s:t], w[s:t])

    def attach_general(self):
        """General-graph partition: exchange the gather lists and attach every pair of ranks that exchanges, in this process."""
        wants = {(r, q): self.strips[r].gpart_wants(q) for r in range(self.world) for q in range(self.world) if q != r}
        pairs = set()
        for (r, q), (idx, slot) in wants.items():
            if idx.size:
                self.strips[q].gpart_set_exports(r, idx, slot)
                pairs.add((r, q)); pairs.add((q, r))
        for (r, q) in sorted(pairs):
            self.strips[r].gpart_attach_local(q, self.strips[q])

    def run(self, iterations, rewards=None):
        import threading
        errs = []

        def work(be):
            try:
                be.run(iterations) if rewards is None else be.run_with_rewards(rewards)
            except Exception as exc:  # noqa: BLE001
                errs.append(exc)
        ts = [threading.Thread(target=work, args=(be,)) for be in self.strips]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        if errs:
            raise errs[0]

    def spike_events(self):
        """The whole lattice's spike events (SNN_OPT_UPDATE_SPIKE_EVENTS on every strip), the ranks' lists merged step by step."""
        return merge_spike_events([be.spike_events() for be in self.strips], self.rows, self.cols)

    def graph_csr(self):
        """Whole-lattice CSR (global presynaptic indices) assembled from the strips."""
        import numpy as np
        rps, pres, ws, base = [np.zeros(1, np.uint64)], [], [], 0
        for be in self.strips:
            rp, pre, w = be.get_connection_csr()
            rps.append(rp[1:] + base)
            pres.append(pre); ws.append(w)
            base += int(rp[-1])
        return np.concatenate(rps), np.concatenate(pres), np.concatenate(ws)
