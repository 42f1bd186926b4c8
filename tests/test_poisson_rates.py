"""Poisson arrivals at a rate per intersection and lane (``BatchedScene.reset_poisson(rates)``,
``pve_reset_poisson_rates``) and the density sweep on generated traffic (``evaluate.evaluate_poisson``).

The stream differs from the one-rate stream only in the mean headway of each lane, so the checks are those of
tests/test_poisson_arrivals.py with rates that differ between lanes and intersections: the mirror, table twins fed
``to_spawn_ticks(poisson_arrivals(..., rates))`` bit for bit on every tick, set_state, sharding and refusals.  Equal
rates must give the traffic of the one-rate reset bit for bit.  Each scene test runs on the emulation of the kernel
source and, marked ``gpu``, on the CUDA build; the launch modes that exist on the device only run on the GPU only.
"""
import ctypes as C
import math
import os

import numpy as np
import pytest
import torch

import parity as P
import test_poisson_arrivals as TP
from pve_mcc_for_unsignalized_intersection_b200 import _native as N
from pve_mcc_for_unsignalized_intersection_b200.arrivals import poisson_arrivals, to_spawn_ticks

GPU = pytest.mark.gpu
BACKENDS = ["emul", pytest.param("cuda", marks=GPU)]
GEOMETRIES = [12, 4, 8]


def spread_rates(B, lanes, lo, hi, seed=0):
    """Rates in [lo, hi] veh/h that differ between every lane and intersection."""
    return np.round(np.random.default_rng(seed).uniform(lo, hi, size=(B, lanes)), 1)


# ---- the mirror ---------------------------------------------------------------------------------------------------
def test_mirror_uniform_array_equals_scalar():
    for lanes in GEOMETRIES:
        a, da = poisson_arrivals(5, 900, 40, seed=3, first_env=11, lanes=lanes)
        for r in (np.full((5, lanes), 900.0), np.full(lanes, 900.0), np.full((5, 1), 900.0)):
            b, db = poisson_arrivals(5, r, 40, seed=3, first_env=11, lanes=lanes)
            assert np.array_equal(a.view(np.int64), b.view(np.int64)) and np.array_equal(da, db)


def test_mirror_reads_rates_like_reset_poisson():
    """[n_envs] is one rate per intersection in the mirror too; a 1-D array is refused when n_envs == lanes."""
    r = np.array([200.0, 700.0, 1300.0, 2000.0, 450.0])
    a, _ = poisson_arrivals(5, r, 30, seed=9)
    b, _ = poisson_arrivals(5, r[:, None], 30, seed=9)
    assert np.array_equal(a.view(np.int64), b.view(np.int64))
    for k in range(5):
        c, _ = poisson_arrivals(1, r[k], 30, seed=9, first_env=k)
        assert np.array_equal(a[k:k + 1].view(np.int64), c.view(np.int64))
    with pytest.raises(ValueError):
        poisson_arrivals(4, np.full(4, 900.0), 30, seed=9, lanes=4)
    with pytest.raises(ValueError):
        poisson_arrivals(5, np.full(3, 900.0), 30, seed=9)


def test_mirror_each_lane_at_its_own_rate():
    """Rates 200, 600 and 1 200 on the lanes of one call: each lane's headways pass the KS / mean-rate check of
    test_poisson_arrivals.test_headway_distribution at its own rate."""
    from scipy import stats
    h0 = 1.0
    rates = np.array([200.0, 600.0, 1200.0] * 4)
    sec, _ = poisson_arrivals(48, rates, 1500, seed=777, min_headway=h0)
    head = np.diff(np.concatenate([np.zeros((sec.shape[0], 1, sec.shape[2])), sec], axis=1), axis=1)
    for rate in (200.0, 600.0, 1200.0):
        lanes = rates == rate
        h = head[:, :, lanes].ravel()
        mean = 3600.0 / rate
        at_h0 = h == h0
        p0 = 1.0 - math.exp(-h0 / mean)
        assert abs(at_h0.mean() - p0) < 5 * math.sqrt(p0 * (1 - p0) / h.size) + 1e-12, (rate, at_h0.mean(), p0)
        ks = stats.kstest(h[~at_h0] - h0, "expon", args=(0, mean))
        assert ks.pvalue > 1e-3, (rate, ks)
        eff = h0 + mean * math.exp(-h0 / mean)
        rate_eff = 3600.0 * h.size / sec[:, -1, lanes].sum()
        assert abs(rate_eff / (3600.0 / eff) - 1) < 0.01, (rate, rate_eff, 3600.0 / eff)


# ---- table twins --------------------------------------------------------------------------------------------------
def _deferred_rates(B, lanes):
    r = np.full((B, lanes), 4000.0)              # a high rate on most lanes of a small class: arrivals are deferred
    r[:, -1] = 700.0
    r[1::2, :-1] *= np.linspace(1.0, 1.5, lanes - 1)
    return r


# name: (B, rates(B, lanes), ticks, scene options, reset options, gpu only)
CASES = {
    "lane12_warmup": (6, lambda B, n: spread_rates(B, n, 200, 1600, 1), 260, dict(), dict(), False),
    "lane12_cold": (6, lambda B, n: spread_rates(B, n, 200, 1600, 2), 200, dict(), dict(warmup=False), False),
    "lane12_per_env": (6, lambda B, n: np.linspace(200, 1200, B)[:, None], 220, dict(), dict(first_env=5), False),
    "lane4": (6, lambda B, n: spread_rates(B, n, 200, 1400, 3), 260, dict(lane_num=4), dict(), False),
    "lane8": (6, lambda B, n: spread_rates(B, n, 200, 1400, 4), 260, dict(lane_num=8), dict(), False),
    "lane8_cold": (6, lambda B, n: spread_rates(B, n, 200, 1400, 5), 200, dict(lane_num=8), dict(warmup=False), False),
    "deferred_96_48": (4, _deferred_rates, 260, dict(veh_cap=96, agent_cap=48), dict(min_headway=0.3), False),
    "lane4_deferred_64": (4, _deferred_rates, 260, dict(lane_num=4, veh_cap=64, agent_cap=64), dict(min_headway=0.3),
                          False),
    "dual_4096": (4096, lambda B, n: spread_rates(B, n, 200, 2400, 6), 140, dict(), dict(seed=11), True),
    "dual_4096_src": (4096, lambda B, n: spread_rates(B, n, 200, 2400, 7), 140,
                      dict(neighbour_sources=True, factored_obs=True), dict(), True),
    "class_576_416": (2, lambda B, n: spread_rates(B, n, 1200, 2400, 8), 260, dict(veh_cap=576, agent_cap=416),
                      dict(min_headway=0.4), True),
}


def _case_params():
    out = []
    for name, c in CASES.items():
        for be in ("emul", "cuda"):
            if c[5] and be == "emul":
                continue
            out.append(pytest.param(be, name, marks=[GPU] if be == "cuda" else [], id="%s-%s" % (be, name)))
    return out


@pytest.mark.parametrize("backend,name", _case_params())
def test_rates_equal_table_twin(backend, name):
    B, rates_of, ticks, opts, ropts, _ = CASES[name]
    ropts = dict(ropts)
    seed = ropts.pop("seed", 2024)
    rates = rates_of(B, opts.get("lane_num", 12))
    pz, tb = TP.twins(backend, B, rates, seed, ticks, **opts, **ropts)
    TP.assert_states_equal(pz.get_state(), tb.get_state(), name + " after reset")
    state_every = 20 if B > 64 else 1
    big = 0
    rng = np.random.default_rng(1)
    for t in range(ticks):
        ctrl = pz.control_mask()
        big = max(big, int(ctrl.sum(dim=1).max()))
        act = P.to_device_actions(pz, P.random_actions(rng, ctrl.cpu().numpy()))
        oa, ob = pz.step(act), tb.step(act.clone())
        TP.assert_outputs_equal(oa, ob, "%s tick %d" % (name, t))
        if (t + 1) % state_every == 0 or t == ticks - 1:
            TP.assert_states_equal(pz.get_state(), tb.get_state(), "%s tick %d" % (name, t))
    TP.assert_stats_equal(pz, tb, name)
    assert int(pz.get_state()["id_seq"].sum()) > B
    if "deferred" in name:
        assert pz.stats()["overflow"] > 0
    if name.startswith("dual"):
        assert pz.launch_info["dual"] and big > 64, big


@GPU
def test_rates_pipelined_host_path_and_rollout():
    """pve_step_host_async and pve_rollout on a per-lane-rate scene and its table twin."""
    from pve_mcc_for_unsignalized_intersection_b200.actor import ActorWeights, BatchedActor
    B, seed, ticks = 512, 8, 120
    pz, tb = TP.twins("cuda", B, spread_rates(B, 12, 200, 2000, 9), seed, 2 * ticks + 20)
    pairs = [s.make_async_buffers(factored=True) for s in (pz, tb)]
    rng = np.random.default_rng(3)
    act_host = torch.zeros(B, pz.veh_cap, dtype=torch.float32).pin_memory()
    for t in range(ticks):
        if t >= 3:
            (na, ha), (nb, hb) = pz.host_wait(), tb.host_wait()
            assert na == nb
            for f in ("packed", "row0_out", "prev_row0", "obs_src"):
                assert torch.equal(TP.bits(getattr(ha, f)[:na]), TP.bits(getattr(hb, f)[:nb])), (t, f)
            assert torch.equal(ha.agent_offset, hb.agent_offset)
        torch.cuda.current_stream().synchronize()
        act_host.copy_(torch.from_numpy(P.random_actions(rng, pz.control_mask().cpu().numpy())))
        for k, s in enumerate((pz, tb)):
            s.step_host_async(act_host, pairs[k][t % 3], copy_factored=True)
    for _ in range(3):
        (na, ha), (nb, hb) = pz.host_wait(), tb.host_wait()
        assert na == nb and torch.equal(ha.packed[:na], hb.packed[:nb])
    TP.assert_states_equal(pz.get_state(), tb.get_state(), "after the pipelined path")
    actor = BatchedActor(ActorWeights.random(0))
    actor.rollout(pz, ticks)
    actor.rollout(tb, ticks)
    TP.assert_outputs_equal(pz.out, tb.out, "last rollout tick")
    TP.assert_states_equal(pz.get_state(), tb.get_state(), "after pve_rollout")
    TP.assert_stats_equal(pz, tb, "after pve_rollout")


# ---- against the one-rate reset, set_state, sharding, mode switches -------------------------------------------------
@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("lane_num", GEOMETRIES)
def test_uniform_array_equals_scalar_reset(backend, lane_num):
    B, rate, seed = 6, 1100, 41
    a, b = TP.make(backend, B, lane_num=lane_num), TP.make(backend, B, lane_num=lane_num)
    a.reset_poisson(np.full((B, lane_num), float(rate)), seed, first_env=3)
    b.reset_poisson(rate, seed, first_env=3)
    TP.assert_states_equal(a.get_state(), b.get_state(), "after reset")
    TP.run_twins(a, b, 200, what="lane_num %d" % lane_num)


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("lane_num", GEOMETRIES)
def test_set_state_mid_rollout_continues_bit_for_bit(backend, lane_num):
    B, seed = 6, 31
    rates = spread_rates(B, lane_num, 300, 1800, 10)
    a = TP.make(backend, B, lane_num=lane_num)
    a.reset_poisson(rates, seed)
    rng = np.random.default_rng(2)
    for _ in range(150):
        a.step(P.to_device_actions(a, P.random_actions(rng, a.control_mask().cpu().numpy())))
    st = a.get_state()
    assert st["veh_rec"].max() > 5
    b = TP.make(backend, B, lane_num=lane_num)
    b.reset_poisson(rates, seed)
    b.set_state(st)
    TP.assert_states_equal(b.get_state(), st, "after set_state", skip=("overflow",))
    for t in range(150):
        act = P.to_device_actions(a, P.random_actions(rng, a.control_mask().cpu().numpy()))
        TP.assert_outputs_equal(a.step(act), b.step(act.clone()), "tick %d after set_state" % t)
    TP.assert_states_equal(a.get_state(), b.get_state(), "end", skip=("overflow",))


@pytest.mark.parametrize("backend", BACKENDS)
def test_sharded_batches_see_the_same_traffic(backend):
    B, seed, ticks = 8, 99, 150
    rates = spread_rates(B, 12, 200, 1800, 11)
    whole = TP.make(backend, B)
    halves = [TP.make(backend, B // 2), TP.make(backend, B // 2)]
    whole.reset_poisson(rates, seed)
    for k, h in enumerate(halves):
        lo = k * B // 2
        h.reset_poisson(rates[lo:lo + B // 2], seed, first_env=lo)
    rng = np.random.default_rng(4)
    for t in range(ticks):
        act = P.random_actions(rng, whole.control_mask().cpu().numpy())
        ow = whole.step(P.to_device_actions(whole, act))
        oh = [h.step(P.to_device_actions(h, act[k * B // 2:(k + 1) * B // 2])) for k, h in enumerate(halves)]
        n0 = oh[0].n_agents
        assert ow.n_agents == n0 + oh[1].n_agents, t
        for f in ("obs", "reward", "status", "jerk_sum", "cpv"):
            a = getattr(ow, f)[:ow.n_agents]
            b = torch.cat([getattr(oh[0], f)[:n0], getattr(oh[1], f)[:oh[1].n_agents]])
            assert torch.equal(TP.bits(a), TP.bits(b)), (t, f)
        sw, s0, s1 = whole.get_state(), halves[0].get_state(), halves[1].get_state()
        for k in sw:
            assert np.array_equal(np.asarray(sw[k]), np.concatenate([s0[k], s1[k]])), (t, k)


@pytest.mark.parametrize("backend", BACKENDS)
def test_mode_switches(backend):
    """Per-lane rates -> one rate -> table -> other per-lane rates on one handle: each reset behaves like a fresh scene
    of its kind."""
    B, ticks = 6, 120
    r1, r2 = spread_rates(B, 12, 200, 1800, 12), spread_rates(B, 12, 2000, 3000, 13)
    tabs = TP.table_for(B, 900, 3, ticks)[0]
    resets = [lambda s: s.reset_poisson(r1, 5), lambda s: s.reset_poisson(1300, 6), lambda s: s.reset(tabs),
              lambda s: s.reset_poisson(r2, 7, min_headway=0.5)]
    s = TP.make(backend, B)
    for k, reset in enumerate(resets):
        fresh = TP.make(backend, B)
        reset(s)
        reset(fresh)
        TP.assert_states_equal(s.get_state(), fresh.get_state(), "reset %d" % k)
        TP.run_twins(s, fresh, ticks, seed=k, state_every=10, what="reset %d" % k)


# ---- refusals -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("backend", BACKENDS)
def test_refusals(backend):
    B = 4
    s = TP.make(backend, B)
    p = N.PvePoisson(1, 0.0, 1.0, 0)
    for bad in (float("nan"), float("inf"), 0.0, -300.0):
        for b, i in ((0, 0), (3, 11), (2, 5)):
            rates = np.full((B, 12), 900.0)
            rates[b, i] = bad
            with pytest.raises(ValueError, match="intersection %d, lane %d" % (b, i)):
                s.reset_poisson(rates, 1)
            rc = s.lib.pve_reset_poisson_rates(s._h, C.byref(p), rates.ctypes.data, 1, s._stream())
            assert rc == -1, (bad, b, i, rc)
            msg = s.lib.pve_last_error(s._h).decode()
            assert msg.startswith("pve_reset_poisson_rates") and "intersection %d, lane %d" % (b, i) in msg, msg
    assert s.lib.pve_reset_poisson_rates(s._h, C.byref(p), None, 1, s._stream()) == -1
    assert "rates_host" in s.lib.pve_last_error(s._h).decode()
    ok = np.full((B, 12), 900.0)
    assert s.lib.pve_reset_poisson_rates(s._h, None, ok.ctypes.data, 1, s._stream()) == -1
    for bad in (dict(min_headway=0.0), dict(first_env=-1), dict(first_env=2**32 - 3)):
        kw = dict(seed=1, min_headway=1.0, first_env=0)
        kw.update(bad)
        with pytest.raises(ValueError):
            s.reset_poisson(ok, **kw)
        q = N.PvePoisson(kw["seed"], 0.0, kw["min_headway"], kw["first_env"])
        assert s.lib.pve_reset_poisson_rates(s._h, C.byref(q), ok.ctypes.data, 1, s._stream()) == -1, bad
        assert s.lib.pve_last_error(s._h).decode().startswith("pve_reset_poisson_rates: "), bad
    for shape in ((B, 11), (B, 13), (B + 1, 12), (B - 1,), (7,), (2, B, 12), (B, 12, 1)):
        with pytest.raises(ValueError):
            s.reset_poisson(np.full(shape, 900.0), 1)
    s4 = TP.make(backend, 4, lane_num=4)                    # n_envs == lane_num: a 1-D array is ambiguous
    with pytest.raises(ValueError, match="ambiguous|one per intersection or one per lane"):
        s4.reset_poisson(np.full(4, 900.0), 1)
    s4.reset_poisson(np.full((4, 1), 900.0), 1)
    s.reset_poisson(np.full(B, 900.0), 1)                   # [B] and [lane_num] are accepted
    s.reset_poisson(np.full(12, 900.0), 1, first_env=2**32 - B)
    assert s.get_state()["id_seq"].sum() > 0


# ---- the density sweep on generated traffic -----------------------------------------------------------------------
@GPU
def test_evaluate_poisson_equals_evaluate_tables():
    """evaluate_poisson's per-intersection tallies equal those of evaluate_tables fed the mirror's tables of the same
    seed and rates, and each pooled line is format_report of the summed tallies."""
    from pve_mcc_for_unsignalized_intersection_b200.actor import ActorWeights
    from pve_mcc_for_unsignalized_intersection_b200.evaluate import evaluate_poisson, evaluate_tables, format_report
    w = ActorWeights.from_npz(os.path.join(os.path.dirname(__file__), "golden", "actor_agent1.npz"))
    densities, n, ticks, seed = (1200, 600, 200), 2, 1500, 17
    got = evaluate_poisson(w, densities=densities, envs_per_density=n, ticks=ticks, seed=seed)
    rates = np.repeat(np.asarray(densities, np.float64), n)[:, None]
    sec, _ = TP.table_for(len(rates), rates, seed, ticks)
    want = evaluate_tables(list(sec), w, ticks=ticks, veh_cap=192, agent_cap=128)
    assert [g["density"] for g in got] == list(densities)
    for k, g in enumerate(got):
        assert g["intersections"] == want[k * n:(k + 1) * n], g["density"]
        pooled = {q: sum(r[q] for r in want[k * n:(k + 1) * n])
                  for q in ("vehicles", "collisions", "passed", "passed_step_total", "jerk_total", "lock_total")}
        assert g["pooled"] == pooled
        assert g["report"] == format_report(**pooled)
        assert pooled["vehicles"] > n
