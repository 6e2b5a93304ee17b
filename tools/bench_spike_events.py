"""Cost of recording spikes on the bench lattice: Izhikevich 3163 x 3163 (10^7 neurons), 8-neighbour grid, electrical synapses
only, the seeded state of bench.py (init_fields, seed 0x5EED).  Three cases over the same number of steps, on one handle that keeps
stepping (warmed up first):
  none    no spike recording
  dense   SNN_OPT_UPDATE_SPIKE_HISTORY: the steps x n u8 raster on the host
  events  SNN_OPT_UPDATE_SPIKE_EVENTS: per step the indices of the neurons that spiked, compacted on the device
Per case:
  us_per_step       device time of the step loop per step (CUDA events on the engine stream; the drains are outside it)
  wall_ms           wall time of run() including every drain
  host_bytes        bytes the recording holds on the host after the run (raster, or step pointers + events)
For events, additionally (torch.profiler, CUDA activity, in a separate run of its own):
  compaction_us_per_chunk   device time of the count kernel, the scan and the scatter kernel per drained chunk
  compaction_GBps           bytes those kernels move per chunk (the staged raster read twice, the events and per-record offsets
                            written) over that time
The card's name and power limit are read in the same process.

    python tools/bench_spike_events.py [--steps 1000] [--out FILE]
"""
import argparse, json, math, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "spiking-neural-networks_b200")):
    sys.path.insert(0, p)
import numpy as np
from snn_b200 import _capi as K
from snn_b200.backend import CudaLatticeBackend
import bench

BUDGET = 256 << 20   # staging bytes per history chunk (engine.cu)
KERNELS = ("spike_event_count_kernel", "graph_row_scan_kernel", "spike_event_scatter_kernel")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def build(rows, cols):
    be = CudaLatticeBackend(K.MODEL_IZH, 0, 0, rows, cols)
    for name, arr in bench.init_fields(np, rows * cols, 0x5EED).items():
        be.set_field(0, name, arr)
    be.connect_grid(0, 1, 1.0)
    be.set_option(K.OPT_ELECTRICAL_SYNAPSE, 1)
    be.set_option(K.OPT_CHEMICAL_SYNAPSE, 0)
    return be


def set_case(be, case):
    be.set_option(K.OPT_UPDATE_SPIKE_HISTORY, int(case == "dense"))
    be.set_option(K.OPT_UPDATE_SPIKE_EVENTS, int(case == "events"))


def run_case(be, case, steps, n):
    set_case(be, case)
    t0 = time.perf_counter()
    ms, launches = be.run_timed(steps)
    wall = (time.perf_counter() - t0) * 1e3
    out = {"us_per_step": 1e3 * ms / steps, "wall_ms": wall, "launches": launches}
    if case == "dense":
        out["host_bytes"] = be.history_len() * n
    elif case == "events":
        sp, nr = be.spike_events()
        assert sp.size == steps + 1
        out["host_bytes"] = sp.nbytes + nr.nbytes
        out["events"] = int(nr.size)
        out["events_per_step"] = nr.size / steps
    else:
        out["host_bytes"] = 0
    be.reset_history()
    set_case(be, "none")
    return out


def compaction(be, steps, n):
    """Device time of the three compaction launches over one run of `steps` steps with events on, per chunk."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    set_case(be, "events")
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        be.run(steps)
        torch.cuda.synchronize()
    sp, nr = be.spike_events()
    be.reset_history()
    set_case(be, "none")
    per = {}
    for ev in prof.key_averages():
        for k in KERNELS:
            if k in ev.key:
                t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
                per[k] = {"us_total": t, "count": ev.count}
    n_words = (n + 31) // 32
    chunk = max(1, min(steps, BUDGET // (4 * n_words)))
    chunks = math.ceil(steps / chunk)
    us = sum(v["us_total"] for v in per.values()) / chunks
    bytes_per_chunk = (2 * 4 * n_words * steps + 4 * nr.size + 4 * steps) / chunks
    return {"chunk_steps": chunk, "chunks": chunks, "kernels": per, "compaction_us_per_chunk": us,
            "compaction_bytes_per_chunk": bytes_per_chunk,
            "compaction_GBps": bytes_per_chunk / (us * 1e-6) / 1e9 if us else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=3163)
    ap.add_argument("--cols", type=int, default=3163)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--out")
    a = ap.parse_args()
    n = a.rows * a.cols
    be = build(a.rows, a.cols)
    be.run_timed(a.warmup)
    res = {"card": card(), "lattice": f"Izhikevich {a.rows}x{a.cols}, radius-1 grid, electrical only, bench.py seeded state",
           "steps": a.steps, "cases": {}}
    # none and events alternate twice (the same handle keeps stepping, so each run sees a later part of the trajectory); the
    # dense raster once, since it holds steps x n bytes on the host
    for case in ("none", "events", "dense", "none", "events"):
        r = run_case(be, case, a.steps, n)
        res["cases"].setdefault(case, []).append(r)
        print(case, json.dumps(r), flush=True)
    res["events_compaction"] = compaction(be, a.steps, n)
    print(json.dumps(res["events_compaction"]), flush=True)
    text = json.dumps(res, indent=1)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
