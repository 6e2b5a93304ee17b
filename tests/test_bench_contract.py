"""bench.py contract, CPU side: the reference arm (the reference algorithm's CPU path = the oracle port, there is no Rust toolchain)
prints exactly one JSON line with the keys the driver reads, and the GPU arm refuses to run without a device instead of falling
back to the CPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--cpu-rows", "96", "--ref-budget-s", "3"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "neuron-steps/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["dtype"] == "f32" and d["data"] == "synthetic"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"] and d["vs_baseline"] is None and d["gpu_launches"] == 0


def test_dump_outputs_writes_a_seeded_sample(tmp_path, monkeypatch):
    """bench.dump_outputs on an oracle lattice (same protocol as CudaLatticeBackend): one float32/float64 .npy per state field plus
    the weights, the values of a fixed sample of neurons and edges, identical on a second call, and within 64 MB at the full
    sample size."""
    import numpy as np
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import bench
    from oracle_api import OracleBackend
    rows = cols = 20
    n = rows * cols
    ob = OracleBackend(4, 0, 0, rows=rows, cols=cols)
    f = bench.init_fields(np, n, 3)
    f["c_m"] = np.full(n, 4.0, np.float32)
    for name, arr in f.items():
        if name not in ("v_init", "w_init"):
            ob.set_field(0, name, arr)
    ob.connect_grid(0, 1, 1.0)
    ob.set_option(0, 1); ob.set_option(1, 1); ob.set_option(2, 1, 0)
    ob.run(30)
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 100)
    bench.dump_outputs(np, ob, str(tmp_path / "a"))
    bench.dump_outputs(np, ob, str(tmp_path / "b"))
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == sorted([nm.replace("$", ".") + ".npy" for nm in bench.STATE_FIELDS] + ["weights.npy"])
    total = 0
    for nm in names:
        a, b = np.load(tmp_path / "a" / nm), np.load(tmp_path / "b" / nm)
        assert a.dtype in (np.float32, np.float64) and a.shape[0] == 100 and np.array_equal(a, b), nm
        total += a.nbytes
    assert total * (1 << 20) // 100 <= 64 << 20
    lft = ob.get_field(0, "last_firing_time")
    got = np.load(tmp_path / "a" / "last_firing_time.npy")
    assert (got >= 0).any() and np.isin(got, lft.astype(np.float64)).all()
    w = ob.get_connection_csr()[2]
    assert (w != 1.0).any() and np.isin(np.load(tmp_path / "a" / "weights.npy"), w).all()


@pytest.mark.gpu
def test_dump_outputs_follow_the_timed_steps(tmp_path):
    """The GPU arm at 264 x 256 (large enough for the bench's window kernel): the same arguments dump the same arrays, and one
    timed step fewer dumps different ones, so the dump is what the last of `--steps` timed steps left."""
    import numpy as np

    def run(tag, steps):
        out = tmp_path / tag
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1", "--iters", "20",
                            "--rows", "264", "--cols", "256", "--no-cpu-baseline", "--no-configs", "--no-e2e", "--no-parity",
                            "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-4000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
        return {p.name: np.load(p) for p in sorted(out.iterdir())}

    a, b, c = run("a", 2), run("b", 2), run("c", 1)
    assert len(a) == 7 and a.keys() == b.keys() == c.keys()
    assert all(np.array_equal(a[k], b[k], equal_nan=True) for k in a)
    assert not np.array_equal(a["current_voltage.npy"], c["current_voltage.npy"])
    assert (a["last_firing_time.npy"] >= 0).any()


def test_gpu_arm_fails_loudly_without_a_device():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a CUDA device is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True,
                       text=True, timeout=300)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


class _StripView:
    """A row strip [row_begin, row_end) of one whole-lattice oracle handle, with the protocol bench.parity_* uses
    (get_field, get_graph_rows with GLOBAL presynaptic indices): stands in for one rank's CudaLatticeBackend on the CPU."""

    def __init__(self, whole, rows, cols, row_begin, row_end):
        self.w, self.rows, self.cols, self.rb, self.re = whole, rows, cols, row_begin, row_end

    def get_field(self, id, name):
        a = self.w.get_field(0, name)
        per = a.size // (self.rows * self.cols)
        return a.reshape(self.rows, self.cols * per)[self.rb:self.re].reshape(-1).copy()

    def get_graph_rows(self, q0, q1):
        import numpy as np
        rp, pre, w = self.w.get_connection_csr(0, 0)
        g0, g1 = self.rb * self.cols + q0, self.rb * self.cols + q1
        s, t = int(rp[g0]), int(rp[g1])
        return (rp[g0:g1 + 1] - rp[g0]).astype(np.uint64), pre[s:t].copy(), w[s:t].copy()


def test_parity_machinery_accepts_the_oracle_and_rejects_a_corrupted_run():
    """bench.py's light-cone parity check (windows straddling every strip boundary, patches assembled from the ranks' pieces, stepped
    on the oracle) run on the CPU: a whole-lattice oracle run viewed as 3 strips must pass; the same run with one voltage or one
    weight nudged inside a window must fail.  Guards the checker itself — a checker that cannot fail proves nothing."""
    import numpy as np
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import bench
    from oracle_api import OracleBackend
    rows, cols, world, k = 70, 45, 3, 5
    n = rows * cols
    ob = OracleBackend(4, 0, 0, rows=rows, cols=cols)
    f = bench.init_fields(np, n, 3)
    f["c_m"] = np.full(n, 4.0, np.float32)    # livelier than the bench's 100 so that STDP has spikes to work with in 40 steps
    for name, arr in f.items():
        if name not in ("v_init", "w_init"):
            ob.set_field(0, name, arr)
    ob.connect_grid(0, 1, 1.0)
    ob.set_option(0, 1); ob.set_option(1, 1); ob.set_option(2, 1, 0)
    ob.run(40)
    bounds = [rows * r // world for r in range(world + 1)]
    wins = bench.parity_windows(rows, cols, bounds, world, k)
    assert sum(any(r0 < bounds[r] < r0 + 16 for r in range(1, world)) for r0, _ in wins) >= world - 1
    views = [_StripView(ob, rows, cols, bounds[r], bounds[r + 1]) for r in range(world)]
    clock0 = ob.get_option(5)
    mine = [bench.parity_collect_before(v, wins, rows, cols, v.rb, v.re, k) for v in views]
    ob.run(k)
    mine = [bench.parity_collect_after(v, m, wins, cols, v.rb, v.re) for v, m in zip(views, mine)]
    rep = bench.parity_compare(np, mine, wins, bounds, rows, cols, world, k, clock0)
    assert rep["ok"] and rep["checked"] == len(wins) and rep["boundaries_covered"] == world - 1, rep
    assert sum(w["learned_weights_in_window"] for w in rep["windows"]) > 0 and sum(w["spiked_in_window_during_check"] for w in rep["windows"]) > 0
    # corrupt one voltage of rank 1's "after" piece of the first boundary window -> must be caught
    import copy
    bad = copy.deepcopy(mine)
    lo, a = bad[1][0]["after"]["current_voltage"]
    a[0, 3, 0] += 0.01
    rep2 = bench.parity_compare(np, bad, wins, bounds, rows, cols, world, k, clock0)
    assert not rep2["ok"] and "current_voltage" in rep2["windows"][0]["mismatch"]
    bad = copy.deepcopy(mine)
    r, rp, pre, w = bad[1][0]["after_edges"][0]
    w[2] += 0.001
    rep3 = bench.parity_compare(np, bad, wins, bounds, rows, cols, world, k, clock0)
    assert not rep3["ok"]
    bad = copy.deepcopy(mine)
    lo, a = bad[0][0]["after"]["last_firing_time"]
    a[-1, 0, 0] += 1
    assert not bench.parity_compare(np, bad, wins, bounds, rows, cols, world, k, clock0)["ok"]
