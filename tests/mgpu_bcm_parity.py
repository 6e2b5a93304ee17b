"""Multi-GPU parity driver for BCM plasticity (launched with torchrun, one rank per GPU; not collected by pytest):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29513 \
        tests/mgpu_bcm_parity.py --rows 203 --cols 97 --steps 150

Every rank steps its partition of a BCM Izhikevich lattice with the BCM rule on.  The ranks exchange spike times and
current_activity through CUDA IPC (the blob offsets of the activity buffers).  Rank 0 also steps the whole lattice on its own GPU,
and the partitions must reproduce it bit for bit: fields, BCM bookkeeping and weights.  --graph random: a random-radius graph whose
edges cross rank boundaries anywhere (general-graph partition).
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "spiking-neural-networks_b200"))

BCM = (0.05, 0.5, 1e-6)   # decay, average_scalar, dt: the parameters of the single-GPU BCM tests


def random_radius_csr(rows, cols, radius, seed=123):
    """For every offset (dr, dc) within the radius, connect with probability 0.6; random weights."""
    n = rows * cols
    g = np.random.default_rng(seed)
    R = int(np.ceil(radius))
    rr, cc = np.divmod(np.arange(n), cols)
    pres, posts, ws = [], [], []
    for dr in range(-R, R + 1):
        for dc in range(-R, R + 1):
            if (dr == 0 and dc == 0) or np.hypot(dr, dc) > radius:
                continue
            ok = (rr + dr >= 0) & (rr + dr < rows) & (cc + dc >= 0) & (cc + dc < cols) & (g.random(n) <= 0.6)
            posts.append(np.nonzero(ok)[0]); pres.append((rr[ok] + dr) * cols + cc[ok] + dc)
            ws.append(g.uniform(0.2, 1.5, int(ok.sum())).astype(np.float32))
    posts, pres, ws = np.concatenate(posts), np.concatenate(pres), np.concatenate(ws)
    order = np.lexsort((pres, posts))
    posts, pres, ws = posts[order], pres[order].astype(np.uint32), ws[order]
    rp = np.zeros(n + 1, np.uint64)
    np.add.at(rp, posts + 1, 1)
    return np.cumsum(rp).astype(np.uint64), pres, ws


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=203)
    ap.add_argument("--cols", type=int, default=97)
    ap.add_argument("--steps", type=int, default=150)
    ap.add_argument("--radius", type=int, default=1)
    ap.add_argument("--no-chem", action="store_true")
    ap.add_argument("--runs", type=int, default=2, help="split the steps over this many run() calls")
    ap.add_argument("--graph", choices=["grid", "random"], default="grid")
    ap.add_argument("--graph-radius", type=float, default=6.0)
    args = ap.parse_args()

    import torch
    import torch.distributed as dist
    from snn_b200 import _capi as K
    from snn_b200.backend import CudaLatticeBackend
    from snn_b200.dist import StripLattice, attach_general

    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rows, cols = args.rows, args.cols
    n = rows * cols
    f32 = np.float32
    rng = np.random.default_rng(77)
    # tonic firing with BCMActivity bookkeeping (the recipe of tests/scenarios.py)
    init = {"current_voltage": rng.uniform(-65, 30, n).astype(f32), "gap_conductance": (10 * rng.uniform(0.5, 1.5, n)).astype(f32),
            "firing_rate_window": rng.choice([1.5, 2.0, 3.25], n).astype(f32), "period": rng.choice([2, 3, 5], n).astype(np.uint32),
            "a": rng.uniform(0.015, 0.03, n).astype(f32), "b": rng.uniform(0.25, 0.36, n).astype(f32),
            "d": rng.uniform(6.0, 9.0, n).astype(f32), "c_m": np.full(n, 2.0, f32)}
    chem = not args.no_chem
    flags = np.zeros((n, 3), np.uint32)
    flags[:, 0] = 1
    csr = random_radius_csr(rows, cols, args.graph_radius) if args.graph == "random" else None

    def configure(be, sl):
        for name, arr in init.items():
            be.set_field(0, name, arr[sl])
        if chem:
            be.set_field(0, "neurotransmitters$flags", flags[sl])
            be.set_field(0, "receptors$flags", flags[sl])
        if csr is None:
            be.connect_grid(0, args.radius, 0.8)
        else:
            rp, pre, w = csr
            q0, q1 = sl.start, sl.stop
            s, t = int(rp[q0]), int(rp[q1])
            if sl.stop - sl.start != n:
                be.set_option(K.OPT_GENERAL_PARTITION, 1)
            be.connect_csr(0, 0, rp[q0:q1 + 1] - rp[q0], pre[s:t], w[s:t])
        be.set_option(K.OPT_ELECTRICAL_SYNAPSE, 1)
        be.set_option(K.OPT_CHEMICAL_SYNAPSE, int(chem))
        be.set_option(K.OPT_DO_PLASTICITY, 1)
        be.set_bcm_plasticity(0, True, *BCM)

    strip = StripLattice(K.MODEL_BCM_IZH, rows, cols, rank, world, device=local)
    sl = slice(strip.row_begin * cols, strip.row_end * cols)
    configure(strip.be, sl)
    if csr is None:
        strip.attach()
    else:
        peers = attach_general(strip.be, rank, world)
        print(f"[rank {rank}] general-graph partition: exchanges with ranks {peers}", flush=True)
    per = [args.steps // args.runs] * args.runs
    per[-1] += args.steps - sum(per)

    def advance(be):
        for k in per:
            be.run(k)

    advance(strip.be)
    names = ["current_voltage", "w_value", "last_firing_time", "is_spiking", "average_activity", "current_activity", "num_spikes",
             "firing_rate_clock"] + (["neurotransmitters$t", "receptors$AMPA$r$kinetics$r"] if chem else [])
    mine = {nm: strip.be.get_field(0, nm) for nm in names}
    _, mine["pre"], mine["weights"] = strip.be.get_connection_csr()
    gathered = [None] * world
    dist.all_gather_object(gathered, mine)
    ok = True
    if rank == 0:
        full = CudaLatticeBackend(K.MODEL_BCM_IZH, 0, 0, rows, cols, device=local)
        configure(full, slice(0, n))
        w0 = full.get_connection_csr()[2].copy()
        advance(full)
        for nm in names:
            want = full.get_field(0, nm)
            got = np.concatenate([g[nm] for g in gathered])
            same = (got == want).all()
            print(f"{nm:32s} {'OK' if same else 'MISMATCH'} ({int((got != want).sum())} of {want.size})")
            ok &= bool(same)
        _, pre2, w2 = full.get_connection_csr()
        gw = np.concatenate([g["weights"] for g in gathered])
        gp = np.concatenate([g["pre"] for g in gathered])
        same = (gp == pre2).all() and (gw == w2).all()
        moved = int((w2 != w0).sum())
        print(f"{'graph (pre, weights)':32s} {'OK' if same else 'MISMATCH'}; weights moved by BCM: {moved} of {w2.size}")
        ok &= bool(same) and moved > 0
        spikes = int((full.get_field(0, "last_firing_time") >= 0).sum())
        print(f"world={world} rows={rows} cols={cols} steps={args.steps} neurons that spiked: {spikes}")
        print("MGPU_BCM_PARITY", "PASS" if ok and spikes > 0 else "FAIL")
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0 and not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
