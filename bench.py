#!/usr/bin/env python
"""bench.py — neuron-steps/s of the lattice stepping hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our CUDA path (default)
    python bench.py --impl reference ...                           # the reference algorithm's CPU path (oracle port)
    python -m torch.distributed.run --nproc-per-node N bench.py --gpus N ...   # one rank per GPU

Workload (config.workload): BASELINE.json configs[4] shape on ONE GPU — Izhikevich 3163x3163 (10^7 neurons), 8-neighbour
Moore grid, electrical + chemical (AMPA, ApproximateNeurotransmitter/ApproximateReceptor) synapses, STDP on, dt = 0.1,
default_impl() neurons with gap_conductance = 10 and V ~ U[v_init, v_th] (SURVEY.md §8d).  For N > 1 the lattice is
(3163*N) x 3163, one 3163-row strip per rank (weak scaling), halos pushed GPU-to-GPU inside the step kernel.

A bench "step" is one `run_lattice(iters)` call = `iters` simulation timesteps over the whole lattice.
`value` times the step loop on the device (CUDA events on the engine's stream, state resident in HBM);
`e2e` times the drop-in call with HOST buffers: every SoA field uploaded from pinned memory, run, state read back.

After the timed region (outside it) every run checks itself against the CPU oracle: 16 x 16 windows — at N > 1 one straddling
EVERY strip boundary — are read with their (16 + 2k)^2 light cones (state + STDP-learned weights) from the live lattice, the
lattice steps k = 12 more timesteps, and the oracle steps the same patches; last_firing_time must be bit-equal, float state equal
to 1e-4.  The line carries `"parity": {"checked": n, "ok": true, ...}`; a mismatch exits non-zero.  At N > 1 the same line also
carries `"strong"`: the SAME 3163-row lattice split over the N GPUs (strong scaling), timed and parity-checked the same way.

`--dump-outputs DIR` (one GPU) writes, right after the timed steps, a seeded sample of the lattice state and weights those steps
left as DIR/<field>.npy (see dump_outputs), so that the outputs of two builds can be compared.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "spiking-neural-networks_b200"))

BYTES_PER_NEURON_STEP = 160.0  # SURVEY.md §8(d), Izhikevich electro-chemical T=1 + STDP, K=8 (derivation in DESIGN.md)
FALLBACK_HBM_GBS = 6650.0      # /opt/skills/guides/B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--rows", type=int, default=3163)
    ap.add_argument("--cols", type=int, default=3163)
    ap.add_argument("--iters", type=int, default=200, help="simulation timesteps per bench step (one run_lattice call)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the step rates of the other BASELINE.json configurations")
    ap.add_argument("--cpu-rows", type=int, default=0, help="side of the CPU lattice (0 = the workload's own rows x cols: same config)")
    ap.add_argument("--ref-budget-s", type=float, default=75.0, help="CPU seconds the timed part of the --impl reference run may take")
    ap.add_argument("--scaling", choices=["weak", "strong"], default="weak",
                    help="weak: rows x cols PER GPU (default, N=1 comparable); strong: ONE rows x cols lattice split over the GPUs")
    ap.add_argument("--no-strong", action="store_true", help="N > 1, weak mode: skip the extra strong-scaling leg")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--parity-steps", type=int, default=12)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a seeded sample of the lattice state and STDP weights to DIR/<name>.npy")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------------ workload
def init_fields(np, n, seed):
    """Synthetic inputs of SURVEY.md §8(d): type defaults, gap_conductance = 10, V ~ U[v_init, v_th]."""
    rng = np.random.default_rng(seed)
    f = {
        "current_voltage": rng.uniform(-65.0, 30.0, n).astype(np.float32),
        "gap_conductance": np.full(n, 10.0, np.float32),
        "w_value": np.full(n, 30.0, np.float32),
        "a": np.full(n, 0.02, np.float32), "b": np.full(n, 0.2, np.float32), "c": np.full(n, -55.0, np.float32),
        "d": np.full(n, 8.0, np.float32), "v_th": np.full(n, 30.0, np.float32), "tau_m": np.full(n, 1.0, np.float32),
        "c_m": np.full(n, 100.0, np.float32), "dt": np.full(n, 0.1, np.float32),
        "v_init": np.full(n, -65.0, np.float32), "w_init": np.full(n, 30.0, np.float32),
        "is_spiking": np.zeros(n, np.uint32), "last_firing_time": np.full(n, -1, np.int32),
    }
    flags = np.zeros((n, 3), np.uint32)
    flags[:, 0] = 1  # AMPA only
    chem = {
        "neurotransmitters$flags": flags.reshape(-1), "receptors$flags": flags.reshape(-1).copy(),
        "neurotransmitters$t": np.zeros(n * 3, np.float32), "neurotransmitters$t_max": np.ones(n * 3, np.float32),
        "neurotransmitters$clearance_constant": np.full(n * 3, 0.01, np.float32),
        "receptors$AMPA_g": np.ones(n, np.float32), "receptors$AMPA_e": np.zeros(n, np.float32),
        "receptors$AMPA$r$kinetics$r": np.zeros(n, np.float32),
    }
    f.update(chem)
    return f


STATE_FIELDS = ["current_voltage", "w_value", "is_spiking", "last_firing_time", "neurotransmitters$t",
                "receptors$AMPA$r$kinetics$r"]


def configure(be, fields):
    for name, arr in fields.items():
        be.set_field(0, name, arr)
    be.connect_grid(0, 1, 1.0)
    be.set_option(0, 1)      # electrical_synapse
    be.set_option(1, 1)      # chemical_synapse
    be.set_option(2, 1, 0)   # do_plasticity (STDP defaults 2, 2, 4.5, 4.5, dt 0.1)


DUMP_SAMPLE = 1 << 20   # neurons and edges kept by --dump-outputs: 44 MB of .npy files in all


def dump_outputs(np, be, out_dir):
    """Write what the timed run_lattice calls left in the lattice, as a caller reads it back: every STATE_FIELDS array and the
    STDP-learned in-edge weights (CSR order).  The whole state of the default workload is about 0.64 GB, so a fixed seeded sample
    of neurons and of edges is kept; the inputs are seeded too, so two builds run with the same arguments compare array for
    array.  Floating-point fields stay float32, integer fields are written as float64 (exact)."""
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(0xD1FF)
    n = be.size()
    cells = np.sort(rng.choice(n, size=min(n, DUMP_SAMPLE), replace=False))
    for nm in STATE_FIELDS:
        a = be.get_field(0, nm).reshape(n, -1)[cells]
        a = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
        np.save(os.path.join(out_dir, nm.replace("$", ".") + ".npy"), a if nm in PER3 else a[:, 0])
    w = be.get_connection_csr()[2]
    edges = np.sort(rng.choice(w.size, size=min(w.size, DUMP_SAMPLE), replace=False))
    np.save(os.path.join(out_dir, "weights.npy"), w[edges])


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU path
def cpu_oracle_run(rows, cols, iters, steps, warmup, parallel, threads):
    """The reference algorithm's CPU path (oracle port: C restatement with array storage — an upper bound on the Rust
    path's speed, BASELINE.md §4) on the workload or a bounded sample of it.  Returns (neuron-steps/s, s per step)."""
    import numpy as np
    os.environ["OMP_NUM_THREADS"] = str(threads)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from oracle_api import OracleBackend
    n = rows * cols
    ob = OracleBackend(4, 0, 0, rows=rows, cols=cols)
    f = init_fields(np, n, 0x5EED)
    for name, arr in f.items():
        if name in ("v_init", "w_init"):
            continue
        ob.set_field(0, name, arr)
    ob.connect_grid(0, 1, 1.0)
    ob.set_option(0, 1); ob.set_option(1, 1); ob.set_option(2, 1, 0); ob.set_option(6, int(parallel))
    for _ in range(warmup):
        ob.run(iters)
    t0 = time.perf_counter()
    for _ in range(steps):
        ob.run(iters)
    dt = time.perf_counter() - t0
    ob.close()
    return n * iters * steps / dt, dt / steps


def reference_arm(args):
    """The reference's own CPU implementation of the path on the box's host cores, on THIS arm's configuration (3163 x 3163,
    same synapses / STDP): every bench step is `iters` whole-lattice timesteps, iters sized so the run ends within minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    rows, cols = (args.cpu_rows, args.cpu_rows) if args.cpu_rows else (args.rows, args.cols)
    same = rows == args.rows and cols == args.cols
    # calibrate on a small lattice (cache-friendly, so it over-estimates the rate: the budget errs on the short side)
    rate, _ = cpu_oracle_run(min(rows, 512), min(cols, 512), 2, 1, 0, True, cores)
    budget = args.ref_budget_s / max(1, args.steps + args.warmup)
    iters = max(1, min(args.iters, int(0.3 * rate * budget / (rows * cols))))
    value, per_step = cpu_oracle_run(rows, cols, iters, args.steps, args.warmup, True, cores)
    sample = (f"{rows}x{cols} Izhikevich lattice ({'the workload itself' if same else 'bounded sample'}: same synapses/STDP), "
              f"{iters} timestep(s) per step, OpenMP gather on {cores} threads")
    line = {
        "impl": "reference", "metric": "neuron-steps/s (Izhikevich lattice)", "value": value, "unit": "neuron-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.gpus, iters_override=iters, sample=sample),
        "cpu_baseline": {"value": value, "unit": "neuron-steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "neuron-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "Rust reference cannot be built here (no rustc/cargo): this is the C oracle port of its CPU algorithm, "
                "gather phase parallel like `parallel = true`, neuron/STDP phase serial (neuron/mod.rs:775-808, 954-982)",
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world, iters_override=None, sample=None, strong=False):
    rows_per = args.rows if not strong else None
    cfg = {
        "workload": "Izhikevich lattice, 8-neighbour Moore grid, electrical + chemical(AMPA) synapses, STDP, dt=0.1 "
                    "(BASELINE.json configs[4] shape)",
        "rows_per_gpu": rows_per if rows_per is not None else f"{args.rows // world}..{-(-args.rows // world)}", "cols": args.cols,
        "neurons_per_gpu": args.rows * args.cols if not strong else args.rows * args.cols // world,
        "global_rows": args.rows * world if not strong else args.rows, "timesteps_per_step": iters_override or args.iters,
        "partition": "row strips, halo pushed over NVLink peer memory inside the step kernel" if world > 1 else "single GPU",
        "l2": "per-step working set ~1.7 GB per GPU >> 126 MB L2 (no flush needed)" if not strong or world == 1 else
              f"per-step working set ~{1700 // world} MB per GPU (larger than the 126 MB L2 up to N = 8)",
    }
    if sample:
        cfg["sample"] = sample
    return cfg


# ------------------------------------------------------------------------------------------------ parity (outside the timed region)
PARITY_STATE = ["current_voltage", "w_value", "is_spiking", "last_firing_time", "neurotransmitters$t", "receptors$AMPA$r$kinetics$r"]
PARITY_PARAMS = ["gap_conductance", "a", "b", "c", "d", "v_th", "tau_m", "c_m", "dt", "neurotransmitters$t_max",
                 "neurotransmitters$clearance_constant", "receptors$AMPA_g", "receptors$AMPA_e"]
PER3 = {"neurotransmitters$t", "neurotransmitters$t_max", "neurotransmitters$clearance_constant"}


def parity_windows(rows_g, cols, bounds, world, k):
    """16 x 16 windows: one straddling EVERY strip boundary (columns alternate left edge / middle / right edge), plus the lattice
    corners and centre.  Returns [(r0, c0)]."""
    h = 16
    wins = []
    col_choices = [0, max(0, cols // 2 - 5), max(0, cols - h)]
    for r in range(1, world):
        wins.append((max(0, min(rows_g - h, bounds[r] - h // 2)), col_choices[r % 3]))
    wins += [(0, 0), (max(0, rows_g - h), max(0, cols - h)), (max(0, rows_g // 2 - 3), max(0, cols // 2 + 7))]
    out = []
    for w in wins:
        if w not in out:
            out.append(w)
    return out


def _cut(nm, arr, cols, row_begin, row_end, ra, rb, ca, cb):
    per = 3 if nm in PER3 else 1
    a = arr.reshape(row_end - row_begin, cols, per)
    lo, hi = max(ra, row_begin), min(rb, row_end)
    return None if lo >= hi else (lo, a[lo - row_begin:hi - row_begin, ca:cb].copy())


def parity_collect_before(be, wins, rows_g, cols, row_begin, row_end, k, h=16):
    """This rank's pieces of every (h+2k)^2 patch: state, parameters and in-edge rows (global presynaptic indices, live weights)."""
    names = PARITY_STATE + PARITY_PARAMS
    full = {nm: be.get_field(0, nm) for nm in names}
    mine = []
    for (r0, c0) in wins:
        ra, rb, ca, cb = max(0, r0 - k), min(rows_g, r0 + h + k), max(0, c0 - k), min(cols, c0 + h + k)
        piece = {"before": {nm: _cut(nm, full[nm], cols, row_begin, row_end, ra, rb, ca, cb) for nm in names}, "edges": []}
        for r in range(max(ra, row_begin), min(rb, row_end)):
            q0 = (r - row_begin) * cols
            piece["edges"].append((r,) + tuple(be.get_graph_rows(q0 + ca, q0 + cb)))
        mine.append(piece)
    return mine


def parity_collect_after(be, mine, wins, cols, row_begin, row_end, h=16):
    after = {nm: be.get_field(0, nm) for nm in PARITY_STATE}
    for (r0, c0), piece in zip(wins, mine):
        piece["after"] = {nm: _cut(nm, after[nm], cols, row_begin, row_end, r0, r0 + h, c0, c0 + h) for nm in PARITY_STATE}
        piece["after_edges"] = []
        for r in range(max(r0, row_begin), min(r0 + h, row_end)):
            q0 = (r - row_begin) * cols
            piece["after_edges"].append((r,) + tuple(be.get_graph_rows(q0 + c0, q0 + c0 + h)))
    return mine


def parity_compare(np, everyone, wins, bounds, rows_g, cols, world, k, clock0, h=16):
    """Rank 0: assemble each patch from the ranks' pieces, step it on the CPU oracle from the same state and clock, compare the
    inner window with what the device produced."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from oracle_api import OracleBackend
    names = PARITY_STATE + PARITY_PARAMS
    report = {"checked": 0, "ok": True, "windows": [], "k": k, "boundaries": world - 1, "boundaries_covered": 0,
              "what": "last_firing_time / is_spiking bit-equal, V / w / t / r and STDP weights to 1e-4 vs the CPU oracle on (16+2k)^2 "
                      "light cones of the live lattice"}
    covered = set()
    for wi, (r0, c0) in enumerate(wins):
        ra, rb, ca, cb = max(0, r0 - k), min(rows_g, r0 + h + k), max(0, c0 - k), min(cols, c0 + h + k)
        pr, pc = rb - ra, cb - ca
        ob = OracleBackend(4, 0, 0, rows=pr, cols=pc)
        fl = np.zeros((pr * pc, 3), np.uint32)
        fl[:, 0] = 1   # AMPA only, as configure() sets it
        ob.set_field(0, "neurotransmitters$flags", fl.reshape(-1))
        ob.set_field(0, "receptors$flags", fl.reshape(-1))
        for nm in names:
            per = 3 if nm in PER3 else 1
            buf = None
            for pieces in everyone:
                got = pieces[wi]["before"][nm]
                if got is None:
                    continue
                lo, a = got
                if buf is None:
                    buf = np.zeros((pr, pc, per), a.dtype)
                buf[lo - ra:lo - ra + a.shape[0]] = a
            ob.set_field(0, nm, buf.reshape(-1))
        # the patch's graph: the live in-edges whose presynaptic cell lies inside the patch, with the learned weights
        rows_seen = {}
        for pieces in everyone:
            for (r, rp, pre, w) in pieces[wi]["edges"]:
                rows_seen[r] = (rp, pre, w)
        rp_all = np.zeros(pr * pc + 1, np.uint64)
        pre_all, w_all = [], []
        for r in range(ra, rb):
            rp, pre, w = rows_seen[r]
            for q in range(pc):
                s, t = int(rp[q]), int(rp[q + 1])
                gr, gc = pre[s:t].astype(np.int64) // cols, pre[s:t].astype(np.int64) % cols
                keep = (gr >= ra) & (gr < rb) & (gc >= ca) & (gc < cb)
                pre_all.append(((gr[keep] - ra) * pc + (gc[keep] - ca)).astype(np.uint32))
                w_all.append(w[s:t][keep])
                rp_all[(r - ra) * pc + q + 1] = rp_all[(r - ra) * pc + q] + int(keep.sum())
        ob.connect_csr(0, 0, rp_all, np.concatenate(pre_all), np.concatenate(w_all))
        ob.set_option(0, 1); ob.set_option(1, 1); ob.set_option(2, 1, 0); ob.set_option(5, clock0)
        ob.run(k)
        hit = [r for r in range(1, world) if r0 < bounds[r] < r0 + h]
        covered.update(hit)
        straddles = bool(hit)
        res = {"r0": r0, "c0": c0, "straddles_boundary": straddles, "ok": True}
        for nm in PARITY_STATE:
            per = 3 if nm in PER3 else 1
            want = ob.get_field(0, nm).reshape(pr, pc, per)[r0 - ra:r0 - ra + h, c0 - ca:c0 - ca + h]
            got = np.zeros_like(want)
            for pieces in everyone:
                g = pieces[wi]["after"][nm]
                if g is not None:
                    got[g[0] - r0:g[0] - r0 + g[1].shape[0]] = g[1]
            if nm in ("last_firing_time", "is_spiking"):
                good = bool((got == want).all())
            else:
                good = bool(np.allclose(got, want, rtol=1e-4, atol=1e-4))
            if not good:
                res["ok"] = False
                res.setdefault("mismatch", []).append(nm)
        # STDP-learned weights of the window's in-edges
        orp, opre, ow = ob.get_connection_csr(0, 0)
        changed = 0
        for pieces in everyone:
            for (r, rp, pre, w) in pieces[wi]["after_edges"]:
                for q in range(min(h, cols - c0)):
                    pq = (r - ra) * pc + (c0 + q - ca)
                    s, t = int(orp[pq]), int(orp[pq + 1])
                    s2, t2 = int(rp[q]), int(rp[q + 1])
                    gr, gc = pre[s2:t2].astype(np.int64) // cols, pre[s2:t2].astype(np.int64) % cols
                    same = (t2 - s2 == t - s) and bool(((gr - ra) * pc + (gc - ca) == opre[s:t]).all())
                    if not same or not np.allclose(w[s2:t2], ow[s:t], rtol=1e-4, atol=1e-5):
                        res["ok"] = False
                        res.setdefault("mismatch", []).append(f"weights of cell ({r},{c0 + q})")
                    changed += int((w[s2:t2] != 1.0).sum())
        lft = ob.get_field(0, "last_firing_time").reshape(pr, pc)[r0 - ra:r0 - ra + h, c0 - ca:c0 - ca + h]
        res["learned_weights_in_window"] = changed
        res["spiked_in_window_during_check"] = int((lft >= clock0).sum())
        ob.close()
        report["windows"].append(res)
        report["checked"] += 1
        report["ok"] = report["ok"] and res["ok"]
    report["boundaries_covered"] = len(covered)
    report["clock"] = [int(clock0), int(clock0 + k)]
    return report


def parity_check(np, be, rows_g, cols, row_begin, row_end, rank, world, k, gather):
    """Light-cone check of the LIVE lattice against the CPU oracle.  Every rank cuts the pieces of the (16+2k)^2 patches it owns
    out of its strip, all ranks step k timesteps, the inner windows are read again; rank 0 compares (parity_compare)."""
    from snn_b200 import _capi as K
    lib = K.load_library()
    bounds = [lib.snn_partition_begin(rows_g, world, r) for r in range(world + 1)]
    wins = parity_windows(rows_g, cols, bounds, world, k)
    clock0 = be.get_option(K.OPT_INTERNAL_CLOCK)
    mine = parity_collect_before(be, wins, rows_g, cols, row_begin, row_end, k)
    be.run(k)
    mine = parity_collect_after(be, mine, wins, cols, row_begin, row_end)
    everyone = gather(mine)
    if rank != 0:
        return None
    return parity_compare(np, everyone, wins, bounds, rows_g, cols, world, k, clock0)


# ------------------------------------------------------------------------------------------------ our arm
def measure_lattice(args, np, torch, dist, K, rows_g, rank, world, local_rank, strong, do_e2e):
    """Build the (strip of the) lattice, time `steps` run_lattice(iters) calls, check parity, measure e2e.  Returns a dict."""
    from snn_b200.backend import CudaLatticeBackend
    from snn_b200.dist import StripLattice
    cols, iters = args.cols, args.iters

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    if world > 1:
        strip = StripLattice(K.MODEL_IZH, rows_g, cols, rank, world, device=local_rank)
        be, row_begin, row_end = strip.be, strip.row_begin, strip.row_end
    else:
        strip, be, row_begin, row_end = None, CudaLatticeBackend(K.MODEL_IZH, 0, 0, rows_g, cols, device=local_rank), 0, rows_g
    n_local = (row_end - row_begin) * cols
    fields = init_fields(np, n_local, 0x5EED + rank)
    configure(be, fields)
    if strip is not None:
        strip.attach()

    for _ in range(args.warmup):
        be.run_timed(iters)
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    t0 = time.perf_counter()
    dev_ms, launches = 0.0, 0
    for _ in range(args.steps):
        ms, nl = be.run_timed(iters)
        dev_ms += ms
        launches += nl
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    t = torch.tensor([dev_ms, wall * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms_max, wall_ms_max = t.tolist()
    spikes = int((be.get_field(0, "last_firing_time") >= 0).sum())
    out = {"be": be, "fields": fields, "n_local": n_local, "dev_ms": dev_ms_max, "wall_ms": wall_ms_max, "launches": launches,
           "clocks": clocks, "spiked_fraction": spikes / max(1, n_local), "rows_global": rows_g,
           "total_neurons": rows_g * cols, "edges_total": 8 * rows_g * cols - 6 * (rows_g + cols) + 4}
    if args.dump_outputs:
        dump_outputs(np, be, args.dump_outputs)

    # ---- parity vs the CPU oracle on the live lattice (outside every timed region)
    if not args.no_parity:
        def gather(obj):
            if world == 1:
                return [obj]
            got = [None] * world
            dist.all_gather_object(got, obj)
            return got
        out["parity"] = parity_check(np, be, rows_g, cols, row_begin, row_end, rank, world, args.parity_steps, gather)

    # ---- e2e: the drop-in call with host buffers (upload every field from pinned memory, run, read the state back)
    if do_e2e:
        pinned = {k: torch.from_numpy(v).pin_memory().numpy() for k, v in fields.items()}
        outs = {name: torch.from_numpy(np.empty_like(fields[name])).pin_memory().numpy() for name in STATE_FIELDS}
        h2d = sum(v.nbytes for v in pinned.values())
        barrier()
        t1 = time.perf_counter()
        for _ in range(args.e2e_steps):
            ta = time.perf_counter()
            configure(be, pinned)
            tb = time.perf_counter()
            be.run(iters)
            tc = time.perf_counter()
            for name in STATE_FIELDS:
                be.get_field(0, name, out=outs[name])
            td = time.perf_counter()
            if os.environ.get("SNN_BENCH_VERBOSE"):
                print(f"[e2e rank {rank}] upload {1e3 * (tb - ta):.1f} ms, run {1e3 * (tc - tb):.1f} ms, download {1e3 * (td - tc):.1f} ms",
                      file=sys.stderr, flush=True)
        barrier()
        e2e_wall = time.perf_counter() - t1
        tt = torch.tensor([e2e_wall], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        d2h = sum(v.nbytes for v in outs.values())
        out["e2e"] = {"value": out["total_neurons"] * iters * args.e2e_steps / tt.item(), "unit": "neuron-steps/s",
                      "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": args.e2e_steps,
                      "what": "snn_lattice_set_field(all fields, pinned host) + set_graph_grid + run(iters) + get_field(state)"}
    return out


def main():
    args = parse_args()
    sys.dont_write_bytecode = True   # the benchmark leaves the tree as it found it (it may be read-only)
    if args.dump_outputs and (args.impl == "reference" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        raise SystemExit("--dump-outputs writes the lattice of the single-GPU CUDA path: one process, --impl ours")
    if args.impl == "reference":
        return reference_arm(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from snn_b200 import _capi as K

    # stdout carries the one JSON line and nothing else: whatever libraries print while we work (NCCL's "NCCL version ..."
    # banner at the first collective, for one) is sent to stderr at the file-descriptor level; fd 1 comes back for the line
    sys.stdout.flush()
    stdout_fd = os.dup(1)
    os.dup2(2, 1)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    iters = args.iters
    strong_main = args.scaling == "strong" and world > 1
    rows_g = args.rows if (strong_main or world == 1) else args.rows * world

    m = measure_lattice(args, np, torch, dist, K, rows_g, rank, world, local_rank, strong_main, not args.no_e2e)
    be = m.pop("be")
    m.pop("fields")
    neuron_steps = m["total_neurons"] * iters * args.steps
    value = neuron_steps / (m["dev_ms"] * 1e-3)

    strong = None
    if world > 1 and not strong_main and not args.no_strong:
        # strong scaling of the named lattice: the SAME rows x cols lattice split over the N GPUs
        be.close()
        sm = measure_lattice(args, np, torch, dist, K, args.rows, rank, world, local_rank, True, False)
        sm.pop("be").close()
        sm.pop("fields")
        strong = {"value": sm["total_neurons"] * iters * args.steps / (sm["dev_ms"] * 1e-3), "unit": "neuron-steps/s",
                  "global_rows": args.rows, "cols": args.cols, "neurons_per_gpu": sm["total_neurons"] // world,
                  "us_per_timestep": sm["dev_ms"] * 1e3 / (iters * args.steps), "ms_per_step": sm["dev_ms"] / args.steps,
                  "clocks": sm["clocks"], "parity": sm.get("parity"),
                  "what": f"the N=1 workload ({args.rows} x {args.cols}) split into {world} row strips: strong scaling; "
                          f"efficiency = value / (N x the N=1 value of this bench)"}

    ok = True
    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (of measured)"
        else:
            peak, peak_src = FALLBACK_HBM_GBS, "B200_PROFILING.md fallback (of fallback)"
        # per GPU: algorithmic bytes of one launch (160 B x the strip's neurons) / the average launch duration of the step loop
        achieved = BYTES_PER_NEURON_STEP * m["n_local"] * iters * args.steps / (m["dev_ms"] * 1e-3) / 1e9
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp) and world == 1:
            tj = json.load(open(tp))
            traffic = tj.get("step_kernel_dram_bytes_per_launch")
            traffic_src = ("profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of one step_win_kernel launch from an "
                           "`ncu --set full` capture of this workload (" + str(tj.get("source", "see profiles/README.md")) + "); "
                           "not re-measured in this run")
        line = {
            "metric": "neuron-steps/s (Izhikevich lattice)", "value": value, "unit": "neuron-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": m["dev_ms"] / args.steps, "higher_is_better": True,
            "scaling": "strong" if strong_main else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, world, strong=strong_main),
            "synaptic_events_per_s": m["edges_total"] * iters * args.steps / (m["dev_ms"] * 1e-3),
            "us_per_timestep": m["dev_ms"] * 1e3 / (iters * args.steps),
            "wall_ms_per_step": m["wall_ms"] / args.steps,
            "spiked_fraction": m["spiked_fraction"],
            "clocks": m["clocks"], "gpu_launches": m["launches"],
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "frac_of_nominal_8000": achieved / 8000.0,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "kernel": "snn::step_win_kernel<IZHIKEVICH, CHEMG=1, NTREL, STDP, G=3> (csrc/step_win.cu)",
                         "bytes_per_neuron_step": BYTES_PER_NEURON_STEP,
                         "avg_launch_us": m["dev_ms"] * 1e3 / max(1, m["launches"])},
        }
        if "parity" in m and m["parity"] is not None:
            line["parity"] = m["parity"]
            ok = ok and m["parity"]["ok"]
        if strong is not None:
            line["strong"] = strong
            if strong.get("parity") is not None:
                ok = ok and strong["parity"]["ok"]
        if "e2e" in m:
            line["e2e"] = m["e2e"]
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            be.close()
            r = 512
            small, _ = cpu_oracle_run(r, r, 40, 1, 0, True, cores)
            single, _ = cpu_oracle_run(r, r, 20, 1, 0, False, 1)
            rows_c, cols_c = (args.cpu_rows, args.cpu_rows) if args.cpu_rows else (args.rows, args.cols)
            par, per = cpu_oracle_run(rows_c, cols_c, 2, 2, 0, True, cores)
            line["cpu_baseline"] = {
                "value": par, "unit": "neuron-steps/s", "cores": cores, "kind": "port",
                "single_thread_value_512": single, "sample_small": {"value": small, "what": f"{r}x{r} lattice (cache-friendly), 40 timesteps, {cores} threads"},
                "sample": f"{rows_c}x{cols_c} lattice (the workload itself), same model/synapses/STDP, 2 timesteps x 2 (gather phase on {cores} "
                          f"OpenMP threads, update+STDP serial, mirroring parallel=true); oracle port = upper bound on the Rust path",
            }
        if world == 1 and not args.no_configs:
            # BASELINE.json configs[0..3] are parity-test cases, not bench lines; their device step rates ride along for the
            # record (SURVEY.md 8d: C1 / C4 are latency-bound, report us per step).  Never allowed to cost the headline line.
            try:
                be.close()
                sys.path.insert(0, os.path.join(ROOT, "tools"))
                import bench_configs
                line["other_configs"] = bench_configs.measure(cpu=False)
            except Exception as exc:  # noqa: BLE001
                line["other_configs"] = {"error": repr(exc)}
        sys.stdout.flush()
        os.dup2(stdout_fd, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if world > 1:
        flag = torch.tensor([0 if ok else 1], device="cuda")
        dist.broadcast(flag, 0)
        ok = flag.item() == 0
        dist.barrier()
        dist.destroy_process_group()
    if not ok:
        print("bench.py: PARITY MISMATCH against the CPU oracle (see the `parity` object of the line above)", file=sys.stderr)
        sys.exit(3)


if __name__ == "__main__":
    main()
