"""Row-strip partitions stepped on ONE GPU (every strip a handle of this process, snn_lattice_attach_local): the multi-GPU data
path — ghost rows pushed into the neighbour's slab by the step kernel, arrival counters, boundary tiles first, lazy STDP across
the strip boundary, the reward-modulated per-edge kernel's second handshake — checked against the CPU oracle by the
single-GPU test tier.  (tests/mgpu_parity.py and bench.py's `parity` object cover real multi-GPU boxes.)"""
import numpy as np
import pytest

import scenarios as SC
import snn_b200 as S
from snn_b200 import _capi as K
from snn_b200.dist import LocalStrips
from oracle_api import OracleBackend

pytestmark = pytest.mark.gpu
f32 = np.float32


def _oracle(rows, cols):
    return OracleBackend(K.MODEL_IZH, 0, 0, rows=rows, cols=cols)


def _configure(set_field, each, n, chem, stdp, radius, seed):
    rng = np.random.default_rng(seed)
    init = {"current_voltage": rng.uniform(-65, 30, n).astype(f32), "b": rng.uniform(0.25, 0.36, n).astype(f32),
            "gap_conductance": (10 * rng.uniform(0.5, 1.5, n)).astype(f32), "c_m": np.full(n, 4.0, f32)}
    for name, arr in init.items():
        set_field(name, arr, 1)
    if chem:
        flags = np.zeros((n, 3), np.uint32)
        flags[:, 0] = 1
        if chem == "mixed":   # the type sets differ from row to row, also across strip boundaries
            flags[:, 0] = (np.arange(n) // 7) % 2
            flags[:, 2] = 1 - flags[:, 0]
        set_field("neurotransmitters$flags", flags, 3)
        rf = np.ones((n, 3), np.uint32)
        set_field("receptors$flags", rf if chem == "mixed" else flags, 3)

    def opts(be):
        be.connect_grid(0, radius, 0.8)
        be.set_option(K.OPT_ELECTRICAL_SYNAPSE, 1)
        be.set_option(K.OPT_CHEMICAL_SYNAPSE, int(bool(chem)))
        be.set_option(K.OPT_DO_PLASTICITY, int(stdp), 0)
        be.set_plasticity(0, 0.05, 0.04, 4.5, 3.0, 0.1)
    each(opts)


STATE = ["current_voltage", "w_value", "last_firing_time", "is_spiking"]


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("shape,radius,chem,stdp", [((41, 33), 1, "ampa", True), ((29, 18), 2, None, False), ((37, 21), 1, "mixed", True),
                                                    ((30, 40), 1, None, True)])
def test_local_strips_match_the_oracle(world, shape, radius, chem, stdp):
    rows, cols = shape
    n = rows * cols
    strips = LocalStrips(K.MODEL_IZH, rows, cols, world)
    _configure(lambda nm, a, per: strips.set_field(nm, a, per), strips.each, n, chem, stdp, radius, 17)
    strips.attach()
    ob = _oracle(rows, cols)
    _configure(lambda nm, a, per: ob.set_field(0, nm, np.asarray(a).reshape(-1)), lambda fn: fn(ob), n, chem, stdp, radius, 17)
    names = STATE + (["neurotransmitters$t", "receptors$AMPA$r$kinetics$r"] if chem else [])
    done = 0
    for k in (25, 1, 24):     # odd and even step counts, several run calls (pending STDP across calls, halo re-push)
        strips.run(k)
        ob.run(k)
        done += k
        for nm in names:
            got, want = strips.get_field(nm), ob.get_field(0, nm)
            if got.dtype.kind in "iu":
                assert (got == want).all(), (nm, done)
            else:
                np.testing.assert_allclose(got, want, rtol=1e-4, atol=1e-3, err_msg=f"{nm} after {done} steps")
    rp, pre, w = strips.graph_csr()
    orp, opre, ow = ob.get_connection_csr()
    assert (rp == orp).all() and (pre == opre).all()
    np.testing.assert_allclose(w, ow, rtol=1e-4, atol=1e-5)
    assert (ob.get_field(0, "last_firing_time") >= 0).sum() > n // 4
    if stdp:
        assert np.abs(ow - 0.8).max() > 1e-3


def test_local_strips_window_kernel_matches_the_oracle(monkeypatch):
    """Two strips large enough for the window-staged TMA kernel (ghost rows enter the stage through the producer's bulk copies,
    boundary tiles are stepped first), electrical + AMPA + STDP as in the bench workload."""
    rows, cols, world = 2 * 132, 256, 2
    n = rows * cols
    strips = LocalStrips(K.MODEL_IZH, rows, cols, world)
    strips.each(lambda be: be.set_option(K.OPT_HALO_TIMEOUT_MS, 20000))
    _configure(lambda nm, a, per: strips.set_field(nm, a, per), strips.each, n, "ampa", True, 1, 23)
    strips.attach()
    ob = _oracle(rows, cols)
    _configure(lambda nm, a, per: ob.set_field(0, nm, np.asarray(a).reshape(-1)), lambda fn: fn(ob), n, "ampa", True, 1, 23)
    for k in (13, 12):
        strips.run(k)
        ob.run(k)
    for nm in ("last_firing_time", "is_spiking"):
        assert (strips.get_field(nm) == ob.get_field(0, nm)).all(), nm
    for nm in ("current_voltage", "w_value", "neurotransmitters$t", "receptors$AMPA$r$kinetics$r"):
        np.testing.assert_allclose(strips.get_field(nm), ob.get_field(0, nm), rtol=1e-4, atol=1e-3, err_msg=nm)
    np.testing.assert_allclose(strips.graph_csr()[2], ob.get_connection_csr()[2], rtol=1e-4, atol=1e-5)


def test_local_strips_reward_modulated():
    """RewardModulatedLattice on strips: the per-edge kernel reads ghost last_firing_time of both parities (second pair of arrival
    counters); weights, traces and dopamine against the oracle."""
    rows, cols, world = 33, 20, 3
    n = rows * cols
    mod = dict(dopamine=0.0, tau_d=20.0, tau_c=0.05, a_plus=0.1, a_minus=0.08, tau_plus=4.5, tau_minus=3.0, dt=0.1)
    strips = LocalStrips(K.MODEL_IZH, rows, cols, world)
    _configure(lambda nm, a, per: strips.set_field(nm, a, per), strips.each, n, None, False, 1, 29)
    strips.each(lambda be: be.set_reward_modulator(True, True, **mod))
    strips.attach()
    ob = _oracle(rows, cols)
    _configure(lambda nm, a, per: ob.set_field(0, nm, np.asarray(a).reshape(-1)), lambda fn: fn(ob), n, None, False, 1, 29)
    ob.set_reward_modulator(True, True, **mod)
    rewards = np.random.default_rng(5).uniform(-0.3, 0.3, 60).astype(f32)
    strips.run(0, rewards=rewards[:31]); ob.run_with_rewards(rewards[:31])
    strips.run(0, rewards=rewards[31:]); ob.run_with_rewards(rewards[31:])
    assert (strips.get_field("last_firing_time") == ob.get_field(0, "last_firing_time")).all()
    np.testing.assert_allclose(strips.get_field("current_voltage"), ob.get_field(0, "current_voltage"), rtol=1e-4, atol=1e-3)
    w, ow = strips.graph_csr()[2], ob.get_connection_csr()[2]
    np.testing.assert_allclose(w, ow, rtol=1e-4, atol=1e-6)
    assert np.abs(ow - 0.8).max() > 1e-4
    tr = [np.concatenate(x) for x in zip(*[be.connection_traces() for be in strips.strips])]
    otr = ob.connection_traces()
    assert (tr[0] == otr[0]).all()
    np.testing.assert_allclose(tr[1], otr[1], rtol=1e-4, atol=1e-7)
    np.testing.assert_allclose(tr[2], otr[2], rtol=1e-4, atol=1e-7)
    for be in strips.strips:
        assert be.get_reward_modulator()["dopamine"] == pytest.approx(ob.get_reward_modulator()["dopamine"], rel=1e-6)


def test_local_strip_halo_timeout_is_an_error_not_a_hang():
    """A strip whose neighbour never runs must come back with SNN_GPU_WAIT_ERROR (bounded wait), not hang the GPU."""
    strips = LocalStrips(K.MODEL_IZH, 20, 16, 2)
    _configure(lambda nm, a, per: strips.set_field(nm, a, per), strips.each, 320, None, False, 1, 3)
    strips.attach()
    strips.each(lambda be: be.set_option(K.OPT_HALO_TIMEOUT_MS, 100))
    with pytest.raises(S.SnnError) as ei:
        strips.strips[0].run(5)     # strip 1 is never stepped
    assert ei.value.status == 6      # SNN_GPU_WAIT_ERROR


# ------------------------------------------------------------------ general-graph partition (SURVEY 8e, second half)
def _random_radius_csr(rows, cols, seed, radius, p):
    """tests/gpu_accuracy.rs:28-32 style: connect x -> y when x != y, distance <= radius, with probability p; random weights."""
    import scenarios as SC
    conn, w = SC.random_graph(rows, cols, seed, radius=radius, p=p, weights="rand")
    return SC.dense_to_csr(conn, w)


def _configure_general(set_field, each, n, chem, stdp):
    rng = np.random.default_rng(19)
    set_field("current_voltage", rng.uniform(-65, 30, n).astype(f32), 1)
    set_field("b", rng.uniform(0.25, 0.36, n).astype(f32), 1)
    set_field("gap_conductance", (10 * rng.uniform(0.5, 1.5, n)).astype(f32), 1)
    set_field("c_m", np.full(n, 4.0, f32), 1)
    if chem:
        set_field("neurotransmitters$flags", _nt_flags(n, chem), 3)
        set_field("receptors$flags", np.ones((n, 3), np.uint32) if chem == "mixed" else _nt_flags(n, chem), 3)

    def opts(be):
        be.set_option(K.OPT_ELECTRICAL_SYNAPSE, 1)
        be.set_option(K.OPT_CHEMICAL_SYNAPSE, int(bool(chem)))
        be.set_option(K.OPT_DO_PLASTICITY, int(stdp), 0)
        be.set_plasticity(0, 0.05, 0.04, 4.5, 3.0, 0.1)
    each(opts)


def _nt_flags(n, chem):
    flags = np.zeros((n, 3), np.uint32)
    flags[:, 0] = 1
    if chem == "mixed":
        flags[:, 0] = (np.arange(n) // 5) % 2
        flags[:, 2] = 1 - flags[:, 0]
    return flags


def _general_matches_the_oracle(parts, rp, pre, w, chem, stdp):
    """Runs the attached partitions and the CPU oracle side by side and compares state and weights."""
    rows, cols = parts.rows, parts.cols
    n = rows * cols
    ob = _oracle(rows, cols)
    _configure_general(lambda nm, a, per: ob.set_field(0, nm, np.asarray(a).reshape(-1)), lambda fn: fn(ob), n, chem, stdp)
    ob.connect_csr(0, 0, rp, pre, w)
    names = STATE + (["neurotransmitters$t", "receptors$AMPA$r$kinetics$r"] if chem else [])
    for k in (21, 1, 20):
        parts.run(k)
        ob.run(k)
        for nm in names:
            got, want = parts.get_field(nm), ob.get_field(0, nm)
            if got.dtype.kind in "iu" or not (chem or stdp):
                assert (got == want).all(), nm
            else:
                np.testing.assert_allclose(got, want, rtol=1e-4, atol=1e-3, err_msg=nm)
    grp, gpre, gw = parts.graph_csr()
    orp, opre, ow = ob.get_connection_csr()
    assert (grp == orp).all() and (gpre == opre).all()
    np.testing.assert_allclose(gw, ow, rtol=1e-4, atol=1e-5)
    assert (ob.get_field(0, "last_firing_time") >= 0).sum() > n // 4
    if stdp:
        assert np.abs(ow - w).max() > 1e-3


@pytest.mark.parametrize("world", [2, 3, 4])
@pytest.mark.parametrize("shape,radius,chem,stdp", [((12, 9), 2.5, None, False), ((16, 10), 5.0, "ampa", True), ((14, 7), 30.0, "mixed", True)])
def test_general_graph_partition_matches_the_oracle(world, shape, radius, chem, stdp):
    """Contiguous node ranges per rank, random-radius graphs whose edges cross rank boundaries arbitrarily (radius 30 = almost
    all-to-all: every rank reads nodes of every other rank, also of non-neighbouring ranks): gather-list ghosts, per-neuron
    export lists, completion counters.  Electrical-only Izhikevich is bit-exact; chemistry + STDP to 1e-4, rasters exact."""
    rows, cols = shape
    rp, pre, w = _random_radius_csr(rows, cols, 41, radius, 0.6)
    parts = LocalStrips(K.MODEL_IZH, rows, cols, world)
    _configure_general(lambda nm, a, per: parts.set_field(nm, a, per), parts.each, rows * cols, chem, stdp)
    parts.set_graph_csr(rp, pre, w)
    parts.attach_general()
    _general_matches_the_oracle(parts, rp, pre, w, chem, stdp)
    if radius >= 30 and world >= 3:   # non-neighbouring ranks exchange too
        idx, _ = parts.strips[0].gpart_wants(world - 1)
        assert idx.size > 0


def test_refused_general_graph_attach_leaves_both_handles_unchanged():
    """An attach that the peer's layout refuses (here: only one rank has chemistry) maps nothing and freezes neither handle: the
    peer can still allocate its chemical fields, and then the ranks attach and match the oracle."""
    rows, cols, chem, stdp = 16, 10, "ampa", True
    n = rows * cols
    rp, pre, w = _random_radius_csr(rows, cols, 41, 5.0, 0.6)
    parts = LocalStrips(K.MODEL_IZH, rows, cols, 2)
    _configure_general(lambda nm, a, per: parts.set_field(nm, a, per), parts.each, n, None, stdp)
    parts.each(lambda be: be.set_option(K.OPT_CHEMICAL_SYNAPSE, 1))
    parts.set_graph_csr(rp, pre, w)
    flags = _nt_flags(n, chem)
    s0, s1 = parts.strips
    s0.set_field(0, "neurotransmitters$flags", flags[parts.rows_of(0)].reshape(-1))
    with pytest.raises(S.SnnError) as ei:
        s0.gpart_attach_local(1, s1)
    assert ei.value.status == K.SNN_INVALID_ARGUMENT
    s1.set_field(0, "neurotransmitters$flags", flags[parts.rows_of(1)].reshape(-1))
    parts.set_field("receptors$flags", flags, 3)
    parts.attach_general()
    _general_matches_the_oracle(parts, rp, pre, w, chem, stdp)
