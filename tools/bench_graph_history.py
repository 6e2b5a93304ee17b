"""Cost of the graph weight history (update_graph_history / update_connecting_graph_history) on the configurations of
BASELINE.json: C1 Izhikevich 100x100 + STDP, C2 LIF 1000x1000 + STDP (radius-1 stencil, ~8 M edges, 32 MB per record), C4 the
MNIST-shaped network (784 Poisson -> 400 exc <-> 400 inh, STDP) with the connecting history and lattice 1's graph history on.

Recording off and on alternate on the same handle (warmed up first).  Per configuration:
  us_per_step_{off,on}     device time of the step loop (CUDA events on the engine stream; record kernels included, drains not)
  host_ms_per_chunk_{off,on}  wall time of run() minus that device time, per history chunk: with recording on this is the drain
                           of the staged records to the host and their split into blocks
  record_kernel_us         graph_record_kernel's own time per launch (torch.profiler, CUDA activity, in a separate pass)
  record_GBps              bytes the record kernel moves (table weights read incl. padding, records written, row offsets read)
                           over that time, next to the 6547 GB/s copy bandwidth this project measures on the card
The card's name and power limit are read in the same process.

    python tools/bench_graph_history.py [--out FILE]
"""
import json, math, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "spiking-neural-networks_b200"), os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle"),
          os.path.join(ROOT, "tools")):
    sys.path.insert(0, p)
import numpy as np
from snn_b200 import _capi as K
import bench_configs as BC

COPY_GBPS = 6547.0
BUDGET = 256 << 20   # staging bytes per history chunk (engine.cu)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def record_bytes(nnz, rows, slots):
    return 4 * slots + 4 * nnz + 4 * (rows + 1)


def kernel_time_us(run):
    """Mean device time of graph_record_kernel over one call of `run` under torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run()
        torch.cuda.synchronize()
    tot, cnt = 0.0, 0
    for ev in prof.key_averages():
        if "graph_record_kernel" in ev.key:
            tot += getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            cnt += ev.count
    return (tot / cnt if cnt else None), cnt


def measure(name, be, set_flags, steps, rounds, nnz, rows, slots, lattice_handle):
    chunks = math.ceil(steps / max(1, min(steps, BUDGET // max(4 * nnz, 4))))
    res = {"off": [], "on": []}
    host = {"off": [], "on": []}
    launches = {}
    for r in range(rounds):
        for mode in ("off", "on"):
            set_flags(mode == "on")
            t0 = time.perf_counter()
            ms, nl = be.run_timed(steps)
            wall = (time.perf_counter() - t0) * 1e3
            res[mode].append(1e3 * ms / steps)
            host[mode].append((wall - ms) / (chunks if mode == "on" else 1))
            launches[mode] = nl
            if mode == "on":
                h = be.graph_history(0, 0) if lattice_handle else be.graph_history(0, 1)
                assert h.shape[0] == steps, h.shape
                be.reset_history()
    set_flags(True)
    k_us, k_cnt = kernel_time_us(lambda: be.run(min(steps, 16)))
    be.reset_history()
    set_flags(False)
    out = {"nnz_per_record": int(nnz), "record_MB": 4 * nnz / 1e6, "steps": steps, "rounds": rounds, "chunks_on": chunks,
           "us_per_step_off": min(res["off"]), "us_per_step_on": min(res["on"]),
           "us_per_step_off_all": res["off"], "us_per_step_on_all": res["on"],
           "host_ms_per_run_off": min(host["off"]), "host_ms_per_chunk_on": min(host["on"]),
           "launches_off": launches["off"], "launches_on": launches["on"],
           "record_kernel_us": k_us, "record_kernel_launches_profiled": k_cnt}
    b = record_bytes(nnz, rows, slots)
    out["record_kernel_bytes"] = b
    if k_us:
        out["record_GBps"] = b / (k_us * 1e-6) / 1e9
        out["record_fraction_of_copy_bw"] = out["record_GBps"] / COPY_GBPS
    else:
        out["record_kernel_us"] = "not measured (no profiler activity)"
    print(name, json.dumps(out), flush=True)
    return out


def lattice_case(cfg, steps, rounds):
    lat = BC.lattice(None, cfg)
    if cfg == "C1":
        lat.do_plasticity = True
    lat._push_options()
    be = lat._be
    be.run_timed(50)
    rp = lat.graph_csr()[0]
    n, nnz = lat.size, int(rp[-1])
    slots = math.ceil(n / 32) * 8 * 32   # radius-1 stencil: 8 k-rows per slice

    def flags(on):
        be.set_option(K.OPT_UPDATE_GRAPH_HISTORY, int(on))
    return measure(cfg, be, flags, steps, rounds, nnz, n, slots, True)


def network_case(steps, rounds):
    net = BC.network(None, None)
    net.get_lattice(1).update_graph_history = True
    net.update_connecting_graph_history = True
    net.run_lattices(100)
    be = net._be
    be.reset_history()
    nnz = sum(be.connection_nnz(a, b) for a, b in ((0, 1), (1, 2), (2, 1), (1, 1)))
    # the table pads each slice to its widest row (rounded to 4): lattice 1's rows take 784 train edges + up to 400 from lattice 2
    slots = math.ceil(400 / 32) * (784 + 400) * 32 + math.ceil(400 / 32) * 4 * 32

    def flags(on):
        be.set_option(K.OPT_UPDATE_CONNECTING_GRAPH_HISTORY, int(on))
        be.set_option(K.OPT_UPDATE_GRAPH_HISTORY, int(on), 1)
    return measure("C4", be, flags, steps, rounds, nnz, 800, slots, False)


def main():
    out_path = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    res = {"card": card()}
    print("card:", res["card"], flush=True)
    res["C1"] = lattice_case("C1", 1000, 3)
    res["C2"] = lattice_case("C2", 40, 3)
    res["C4"] = network_case(1000, 3)
    txt = json.dumps(res, indent=1)
    print(txt)
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
