"""BCM plasticity on row strips: device time per step of a BCM Izhikevich lattice of 3163 x 3163 neurons (10^7), radius-1
stencil, electrical synapses, BCM on (decay 0.05, average_scalar 0.5, dt 1e-6).

  whole          the lattice as one handle on GPU 0
  strips_N       the same lattice as N row strips driven from this process (LocalStrips(devices=[0 .. N-1])), for every N >= 2
                 that is visible; per step = the slowest strip's device time
  ab             whole lattice, the library under test against a baseline library (--baseline-lib, e.g. the parent commit's
                 build), each round one fresh process per library, alternating
Per step = the device time of the step loop from run_timed (CUDA events on the engine's stream): the step kernel and the BCM
edge kernel of every timestep.  The edge kernel skips edges with no spiking end, so the time depends on the simulated window:
the rounds of `whole` and `strips_N` continue one simulation, while every `ab` round times the same window (steps warmup + 1 ..
warmup + steps from the seeded state).  The card's name, power limit and SM clocks are read in the same call.

    python tools/bench_bcm_partitions.py [--steps 200] [--rounds 3] [--baseline-lib PATH] [--out FILE]
"""
import argparse, json, os, subprocess, sys, threading
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "spiking-neural-networks_b200"))
import numpy as np

ROWS = COLS = 3163
BCM = (0.05, 0.5, 1e-6)
f32 = np.float32


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines() if q.returncode == 0 and q.stdout.strip() else ["unknown"]


def fields(n, seed=7):
    """A tonically firing BCM Izhikevich lattice (the recipe of tests/scenarios.py)."""
    rng = np.random.default_rng(seed)
    return {"current_voltage": rng.uniform(-65, 30, n).astype(f32), "gap_conductance": (10 * rng.uniform(0.5, 1.5, n)).astype(f32),
            "firing_rate_window": rng.choice([1.5, 2.0, 3.25], n).astype(f32), "period": rng.choice([2, 3, 5], n).astype(np.uint32),
            "a": rng.uniform(0.015, 0.03, n).astype(f32), "b": rng.uniform(0.25, 0.36, n).astype(f32),
            "d": rng.uniform(6.0, 9.0, n).astype(f32), "c_m": np.full(n, 2.0, f32)}


def configure(be):
    from snn_b200 import _capi as K
    be.connect_grid(0, 1, 0.8)
    be.set_option(K.OPT_ELECTRICAL_SYNAPSE, 1)
    be.set_option(K.OPT_DO_PLASTICITY, 1, 0)
    be.set_bcm_plasticity(0, True, *BCM)


def whole(steps, rounds, warmup):
    from snn_b200 import _capi as K
    from snn_b200.backend import CudaLatticeBackend
    be = CudaLatticeBackend(K.MODEL_BCM_IZH, 0, 0, ROWS, COLS, device=0)
    for name, a in fields(ROWS * COLS).items():
        be.set_field(0, name, a)
    configure(be)
    be.run_timed(warmup)
    per, launches = [], None
    for _ in range(rounds):
        ms, launches = be.run_timed(steps)
        per.append(1e3 * ms / steps)
    return {"us_per_step": min(per), "us_per_step_all": per, "launches_per_run": launches, "steps": steps}


def strips(world, steps, rounds, warmup):
    from snn_b200 import _capi as K
    from snn_b200.dist import LocalStrips
    parts = LocalStrips(K.MODEL_BCM_IZH, ROWS, COLS, world, devices=list(range(world)))
    for name, a in fields(ROWS * COLS).items():
        parts.set_field(name, a)
    parts.each(configure)
    parts.attach()

    def timed(k):
        out = [None] * world

        def work(r):
            out[r] = parts.strips[r].run_timed(k)
        ts = [threading.Thread(target=work, args=(r,)) for r in range(world)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        return out
    timed(warmup)
    per, per_strip = [], []
    for _ in range(rounds):
        out = timed(steps)
        per_strip.append([1e3 * ms / steps for ms, _ in out])
        per.append(max(per_strip[-1]))
    return {"us_per_step": min(per), "us_per_step_all": per, "us_per_step_per_strip": per_strip, "steps": steps,
            "launches_per_run": [nl for _, nl in out]}


def worker(lib, steps, warmup):
    """One process, one library: the whole lattice, printed as one JSON line."""
    from snn_b200 import _capi as K
    if lib:
        K._lib = K.load_library(lib)
    print("RESULT " + json.dumps(whole(steps, 1, warmup)), flush=True)


def ab(baseline, steps, rounds, warmup):
    libs = {"new": None, "baseline": os.path.abspath(baseline)}
    res = {k: [] for k in libs}
    for _ in range(rounds):
        for name, lib in libs.items():
            cmd = [sys.executable, os.path.abspath(__file__), "--worker", "--steps", str(steps), "--warmup", str(warmup)]
            if lib:
                cmd += ["--lib", lib]
            out = subprocess.run(cmd, capture_output=True, text=True, check=True).stdout
            line = [l for l in out.splitlines() if l.startswith("RESULT ")][0]
            res[name].append(json.loads(line[7:])["us_per_step"])
    return {"us_per_step_new": min(res["new"]), "us_per_step_baseline": min(res["baseline"]),
            "us_per_step_new_all": res["new"], "us_per_step_baseline_all": res["baseline"], "order": "new, baseline per round"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--baseline-lib")
    ap.add_argument("--out")
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--lib")
    a = ap.parse_args()
    if a.worker:
        return worker(a.lib, a.steps, a.warmup)
    import ctypes as C
    from snn_b200 import _capi as K
    cnt = C.c_int32()
    K.check(K.load_library(), K.load_library().snn_device_count(C.byref(cnt)))
    n_dev = cnt.value
    res = {"workload": f"BCM Izhikevich {ROWS} x {COLS}, radius-1 stencil, electrical, BCM decay/average_scalar/dt = {BCM}",
           "cards": card(), "devices_visible": n_dev}
    print(json.dumps(res), flush=True)
    res["whole"] = whole(a.steps, a.rounds, a.warmup)
    print("whole", json.dumps(res["whole"]), flush=True)
    for world in range(2, n_dev + 1):
        res[f"strips_{world}"] = strips(world, a.steps, a.rounds, a.warmup)
        print(f"strips_{world}", json.dumps(res[f"strips_{world}"]), flush=True)
    if n_dev < 2:
        res["strips"] = f"not measured: {n_dev} device visible"
    res["ab"] = ab(a.baseline_lib, a.steps, a.rounds, a.warmup) if a.baseline_lib else "not measured: no --baseline-lib"
    print("ab", json.dumps(res["ab"]), flush=True)
    res["cards_after"] = card()
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
