"""The launch sequence of Engine::run, pinned by the launch count run_timed(k) reports on every step path: one launch per
timestep kernel, per-edge plasticity pass, spike-train step and graph record, plus the end-of-run STDP flush and the halo push of
a partitioned handle.  k = 1 and an odd k (ping-pong parity, the first step of a run has no pending STDP)."""
import math
import threading

import pytest

import scenarios as SC
import snn_b200 as S
from snn_b200 import _capi as K
from snn_b200.dist import LocalStrips
from test_gpu_parity import build_network
from test_gpu_strips import _configure
from test_reward_network import build_reward_network

pytestmark = pytest.mark.gpu

KS = (1, 5)


def _lattice_run(lat, spg=None):
    be = lat._be
    if spg is not None:
        be.set_option(K.OPT_STEPS_PER_GRAPH, spg)

    def run(k):
        lat._push_options()
        return be.run_timed(k)[1]
    return run


def _network_run(net, spg=None):
    net.run_lattices(0)   # pushes the options
    be = net._be
    if spg is not None:
        be.set_option(K.OPT_STEPS_PER_GRAPH, spg)

    def run(k):
        net.run_lattices(0)
        return be.run_timed(k)[1]
    return run


def _stdp_lattice(**kw):
    return SC.build_lattice(None, model="izh", rows=20, cols=24, seed=3, graph="grid", **kw)


@pytest.fixture
def kernel_env(monkeypatch):
    def set_env(tma, win):
        monkeypatch.setenv("SNN_B200_TMA", tma)
        monkeypatch.setenv("SNN_B200_WIN", win)
    return set_env


@pytest.mark.parametrize("stdp", [False, True])
@pytest.mark.parametrize("kernel", ["win", "tma"])
def test_staged_lattice_launches(kernel, stdp, kernel_env):
    kernel_env("2", "1" if kernel == "win" else "0")
    run = _lattice_run(_stdp_lattice(stdp=stdp))
    for k in KS:
        assert run(k) == k + (1 if stdp else 0)   # one persistent kernel per step, the flush


def test_general_lattice_launches(kernel_env):
    kernel_env("0", "0")
    run = _lattice_run(SC.build_lattice(None, model="lif", rows=9, cols=12, seed=5, graph="random", stdp=True, gap=40.0), spg=1)
    for k in KS:
        assert run(k) == k + 1


def test_bcm_lattice_launches():
    lat = SC.build_lattice(None, model="bcm_izh", rows=7, cols=9, seed=4, graph="random", stdp=True)
    lat.plasticity = S.BCM(decay=0.05, average_scalar=0.5, dt=1e-6)
    run = _lattice_run(lat)
    for k in KS:
        assert run(k) == 2 * k   # step kernel + BCM edge kernel, no flush


def test_reward_modulated_lattice_launches():
    lat = SC.build_lattice(None, model="izh", rows=7, cols=9, seed=4, graph="grid", cls=S.RewardModulatedLattice)
    run = _lattice_run(lat)
    for k in KS:
        assert run(k) == 2 * k   # step kernel + reward-modulated edge kernel


@pytest.mark.parametrize("shape,per_step", [((3, 4), 2), ((16, 16), 2)], ids=["general", "two_pass_wide"])
def test_network_with_trains_launches(shape, per_step):
    # general kernel: step + trains; two-pass wide kernel (very wide rows): terms pass + sum pass, the trains ride in the sum pass
    run = _network_run(build_network(None, None, train="rate", stdp=True, st_shape=shape), spg=1)
    for k in KS:
        assert run(k) == per_step * k + 1


def test_reward_modulated_network_launches():
    run = _network_run(build_reward_network(None, None))
    for k in KS:
        assert run(k) == 3 * k   # step, weight pass, trains


@pytest.mark.parametrize("spg", [0, 1, 7])
def test_multi_step_launches(spg):
    run = _lattice_run(SC.build_lattice(None, model="lif", rows=9, cols=12, seed=5, graph="random", stdp=True, gap=40.0), spg=spg)
    for k in KS:
        per_run = 1 if spg == 0 else math.ceil(k / spg)
        assert run(k) == per_run + 1


def test_graph_history_lattice_launches():
    lat = _stdp_lattice(stdp=True, history=False)
    lat.update_graph_history = True
    run = _lattice_run(lat)
    for k in KS:
        # k step kernels, the flush, and k records (steps 1 .. k-1 after the next step kernel, the last one after the flush)
        assert run(k) == 2 * k + 1


def test_graph_history_network_launches():
    net = build_network(None, None, train="rate", stdp=True)
    net.get_lattice(1).update_graph_history = True
    net.update_connecting_graph_history = True
    run = _network_run(net)
    for k in KS:
        assert run(k) == 3 * k + 1   # step, trains and record per step, the flush (a network records before it)


def test_local_strips_launches():
    strips = LocalStrips(K.MODEL_IZH, 20, 16, 2)
    _configure(lambda nm, a, per: strips.set_field(nm, a, per), strips.each, 320, None, True, 1, 3)
    strips.attach()
    for k in KS:
        out = [None] * len(strips.strips)

        def work(r):
            out[r] = strips.strips[r].run_timed(k)[1]
        ts = [threading.Thread(target=work, args=(r,)) for r in range(len(strips.strips))]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        assert out == [k + 2] * len(strips.strips)   # halo push, k step kernels, the flush
