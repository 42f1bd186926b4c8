"""Statistics parity: the per-intersection running statistics of the step kernels (``pve_env_stats_dev``, the float64
``[B, 10]`` array behind ``BatchedScene.env_stats``) and the end-of-rollout counters (``pve_stats``, ``stats()``)
against an independent float64 reduction.

The bench line (agent and vehicle steps), the evaluation report (collisions, jerks, lock events) and the vector that
multi-GPU runs all-reduce all come from these numbers, not from the per-agent rows.  Each check here sums the
reference's quantities tick by tick on the host:

* from the oracle's own per-tick outputs and the state it starts the tick from (``Tally.add_oracle``), or
* where the oracle is too slow or cannot see the rows, from the rows the scene itself delivered, summed in float64
  (``rows_tally``).

Every test runs on the sequential emulation of the kernel source (CPU tier) and, marked ``gpu``, on the CUDA build; the
launch modes that exist on the device only (CTA sizes, the dual-kernel launch, the host paths with pinned buffers, the
pipelined host path, the 256-thread reduction at B > 256, the evaluation driver) run on the GPU only.
"""
import os
import sys

import numpy as np
import pytest
import torch

import parity as P
import test_kernel4_logic_emul as E4
from golden_io import snapshot_to_state
from pve_mcc_for_unsignalized_intersection_b200 import _native as N
from pve_mcc_for_unsignalized_intersection_b200.arrivals import stress_arrivals, synthetic_arrivals
from pve_mcc_for_unsignalized_intersection_b200.scene import BatchedScene

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import make_golden as MG  # noqa: E402  (crafted-state helpers of crafted.npz)

GPU = pytest.mark.gpu
BACKENDS = ["emul", pytest.param("cuda", marks=GPU)]

NAMES = BatchedScene.ENV_STAT_NAMES
Q = {n: q for q, n in enumerate(NAMES)}
FLOAT_STATS = ("passed_jerk_sum", "reward_sum", "reward_sq_sum")
# relative bounds, times sum |x| of the quantity; integer statistics are exact
ORACLE_TOL = {"passed_jerk_sum": 1e-12,      # bit-exact float64 state, only the summation order differs
              "reward_sum": 1e-5, "reward_sq_sum": 1e-5}        # fp32 rewards against float64 ones
ROWS_TOL = {"passed_jerk_sum": 1e-7,         # the rows carry jerk_sum as float32, the kernel sums the float64 state
            "reward_sum": 1e-12, "reward_sq_sum": 1e-12}        # the same fp32 rewards, summed in another order


# ---- reference accumulators ---------------------------------------------------------------------------------------
class Tally:
    """float64 ``[B, 10]`` sums in ``ENV_STAT_NAMES`` order, with the sums of ``|x|`` that scale the tolerances."""

    def __init__(self, B):
        self.B = B
        self.s = np.zeros((B, len(NAMES)))
        self.mag = np.zeros((B, len(NAMES)))

    def add_rows(self, off, n_veh, cpv, status, jerk_sum, reward, lock, removed, q5):
        """One tick: ``off`` the agent offsets, ``n_veh`` the vehicles present when the tick started (before its
        spawns), then the per-agent rows and the per-intersection counters."""
        B = self.B
        env = np.repeat(np.arange(B), np.diff(off))
        per = lambda w: np.bincount(env, weights=np.asarray(w, np.float64), minlength=B)
        r = np.asarray(reward, np.float64)
        jk = np.where((np.asarray(status) & N.ST_FINISHED) != 0, np.asarray(jerk_sum, np.float64), 0.0)
        vals = np.stack([np.diff(off).astype(np.float64), np.asarray(n_veh, np.float64), per(np.asarray(cpv) > 0),
                         np.asarray(lock, np.float64), per(jk), per(r), per(r * r), np.asarray(removed, np.float64),
                         np.ones(B), np.asarray(q5, np.float64)], axis=1)
        self.s += vals
        self.mag += np.abs(vals)
        self.mag[:, Q["passed_jerk_sum"]] += per(np.abs(jk)) - np.abs(vals[:, Q["passed_jerk_sum"]])
        self.mag[:, Q["reward_sum"]] += per(np.abs(r)) - np.abs(vals[:, Q["reward_sum"]])

    def add_oracle(self, st, o):
        """``st``: the oracle's state before ``orc.step``; ``o``: what that step returned."""
        self.add_rows(o["agent_offset"], st["lane_n"].sum(axis=1), o["cpv"], o["status"], o["jerk_sum"], o["reward"],
                      o["lock"], o["n_removed"], o["q5_undefined"])


def rows_tally(tally, n_veh, out):
    """The device-output accumulator: the float32 rows of ``out`` (``StepOutputs``), observations left where they are."""
    n = out.n_agents
    g = lambda t: t.cpu().numpy()
    tally.add_rows(g(out.agent_offset), n_veh, g(out.cpv[:n]), g(out.status[:n]), g(out.jerk_sum[:n]), g(out.reward[:n]),
                   g(out.env_lock), g(out.env_removed), np.zeros(tally.B))


def vehicles_now(scene):
    """Vehicles present in every intersection right now, from the device header's lane counts: the ``vehicle_steps``
    term of the next tick."""
    hdr = scene._wrap(scene.lib.pve_hdr_dev(scene._h), (scene.B, N.HDR_DTYPE.itemsize), torch.uint8, "|u1")
    o = N.HDR_DTYPE.fields["lane_n"][1]
    return hdr[:, o:o + 12].to(torch.int64).sum(dim=1).cpu().numpy()


def env_stats(scene):
    return scene.env_stats().cpu().numpy().astype(np.float64, copy=True)


def compare_stats(got, tally, tol, what, skip=()):
    for q, name in enumerate(NAMES):
        if name in skip:
            continue
        g, w = got[:, q], tally.s[:, q]
        bad = np.abs(g - w) > tol[name] * tally.mag[:, q] if name in FLOAT_STATS else g != w
        if bad.any():
            b = int(np.argmax(bad))
            raise AssertionError("%s: %s of intersection %d is %r, the reference sum is %r (%d intersections differ)"
                                 % (what, name, b, g[b], w[b], int(bad.sum())))


def check_reset_row(scene, warmup):
    """Right after ``reset``: the warm-up tick counts as one env step (and nothing else: the scene is empty), no
    warm-up means all zeros.  Returns the row, subtracted from later readings."""
    es = env_stats(scene)
    want = np.zeros_like(es)
    want[:, Q["env_steps"]] = 1.0 if warmup else 0.0
    np.testing.assert_array_equal(es, want, err_msg="statistics after reset(warmup=%s)" % warmup)
    return es


def check_reduction(scene):
    """``stats()`` (``pve_stats``) = the column sums of ``env_stats()`` plus the header counters of ``get_state()``,
    slot by slot in ``COUNTER_NAMES`` order."""
    s = scene.stats()
    assert list(s) == N.COUNTER_NAMES and len(s) == 16
    es, st = env_stats(scene), scene.get_state()
    for q, name in enumerate(NAMES):
        col = es[:, q]
        if name in FLOAT_STATS:
            assert abs(s[name] - col.sum()) <= 1e-12 * np.abs(col).sum(), (name, s[name], col.sum())
        else:
            assert s[name] == col.sum(), (name, s[name], col.sum())
    for name, key in (("spawned", "id_seq"), ("passed", "passed_veh"), ("passed_step_total", "passed_step_total"),
                      ("overflow", "overflow")):
        assert s[name] == int(st[key].astype(np.int64).sum()), (name, s[name], int(st[key].sum()))
    assert s["reserved0"] == 0 and s["reserved1"] == 0
    return s, es, st


def policy_actions(policy, rng, ctrl, t, fill):
    """uniform: random accelerations (collisions, lock events); brake / mixed: full braking (queues fill the large
    classes), mixed alternating with random ticks once ``fill`` ticks are over."""
    if policy == "uniform" or (policy == "mixed" and t >= fill and t % 2):
        return P.random_actions(rng, ctrl)
    return np.where(ctrl, -3.0, 0.0).astype(np.float32)


def drive(scenes, orc, tabs, ticks, seed, policy="uniform", fill=0, warmup=True, garbage=False, every_tick=None):
    """Reset ``scenes`` and ``orc`` with ``tabs``, drive them with the same actions for ``ticks`` ticks and compare the
    statistics of every scene with the oracle tally after every tick.  ``garbage``: the scenes get random values in the
    slots of uncontrolled vehicles (``zero_uncontrolled_actions``), the oracle the reference driver's zeros.
    Returns the tally and, per scene, the statistics accumulated since the reset."""
    B = tabs.shape[0]
    for sc in scenes:
        sc.reset(tabs, warmup=warmup)
    orc.reset(tabs, warmup=warmup)
    bases = [check_reset_row(sc, warmup) for sc in scenes]
    tally = Tally(B)
    rng = np.random.RandomState(seed)
    for t in range(ticks):
        st = orc.get_state()
        ctrl = (st["flags"] & 1) != 0
        act = policy_actions(policy, rng, ctrl, t, fill)
        dev_act = np.where(ctrl, act, rng.uniform(-3, 3, size=act.shape)).astype(np.float32) if garbage else act
        if every_tick is not None:
            every_tick(t, st)
        o = orc.step(act)
        assert o["overflow"] == 0, "the oracle dropped an arrival: the case leaves its capacity class"
        tally.add_oracle(st, o)
        for sc in scenes:
            sc.step(P.to_device_actions(sc, dev_act))
        for sc, base in zip(scenes, bases):
            compare_stats(env_stats(sc) - base, tally, ORACLE_TOL, "tick %d" % t)
    ref = orc.get_state()
    for sc in scenes:
        P.compare_states(sc.get_state(), ref, "final")
        check_reduction(sc)
    return tally, [env_stats(sc) - base for sc, base in zip(scenes, bases)]


def assert_nontrivial(tally, what):
    tot = tally.s.sum(axis=0)
    for name in ("collided_agent_steps", "lock_events", "removed", "passed_jerk_sum"):
        assert tot[Q[name]] > 0, "%s: no %s in the whole run" % (what, name)


# ---- 2. coverage matrix: every capacity class, CTA size and launch mode against the oracle -------------------------
def mixed_tables(B, rate, seed, rows=48):
    return synthetic_arrivals(B, rate, 45.0, seed=seed, rows=rows)


# name: (tables, ticks, policy, fill, scene options, (vehicles, agents) of the next smaller class, of which some intersection
# must exceed one, gpu only)
CASES = {
    "class_128_80": (lambda: mixed_tables(4, 1400, 3), 300, "uniform", 0, dict(veh_cap=128, agent_cap=80), (96, 64), False),
    "class_128_96": (lambda: mixed_tables(4, 1200, 4), 300, "uniform", 0, dict(veh_cap=128, agent_cap=96), (96, 64), False),
    "class_192_128": (lambda: mixed_tables(4, 2000, 5, rows=60), 300, "uniform", 0, dict(veh_cap=192, agent_cap=128),
                      (128, 96), False),
    "class_384_320": (lambda: stress_arrivals(2, 40.0), 300, "mixed", 200, dict(veh_cap=384, agent_cap=320),
                      (192, 128), False),
    "class_576_416": (lambda: stress_arrivals(1, 60.0, headway=0.7), 420, "mixed", 300, dict(veh_cap=576, agent_cap=416),
                      (384, 320), False),
    "neighbour_sources": (lambda: mixed_tables(4, 1200, 6), 300, "uniform", 0, dict(neighbour_sources=True), (64, 48), False),
    "zero_uncontrolled_actions": (lambda: mixed_tables(4, 1200, 7), 300, "uniform", 0,
                                  dict(zero_uncontrolled_actions=True), (64, 48), False),
}
for _nt in (64, 96, 128, 256, 512):        # CTA sizes of the default class (64 and 96: no team / mover split)
    CASES["threads_%d" % _nt] = (lambda: mixed_tables(4, 1400, 8), 300, "uniform", 0, dict(threads=_nt), (96, 64), True)
CASES["threads_0_class_384_320"] = (lambda: stress_arrivals(2, 40.0, headway=1.2), 300, "mixed", 200,
                                    dict(veh_cap=384, agent_cap=320, threads=0), (192, 128), True)


def _case_params():
    out = []
    for name, case in CASES.items():
        out.append(pytest.param("cuda", name, marks=GPU, id="cuda-" + name))
        if not case[-1]:
            out.insert(len(out) - 1, pytest.param("emul", name, id="emul-" + name))
    return out


@pytest.mark.parametrize("backend,case", _case_params())
def test_statistics_match_the_oracle(backend, case):
    make_tabs, ticks, policy, fill, opts, (min_v, min_a), _ = CASES[case]
    tabs = make_tabs()
    B = tabs.shape[0]
    scene = P.make_scene(backend, B, vm=5, **opts)
    if "veh_cap" in opts:
        assert (scene.veh_cap, scene.agent_cap) == (opts["veh_cap"], opts["agent_cap"])
    orc = P.make_oracle(B, vm=5, veh_cap=scene.veh_cap)
    peak = np.zeros(2, int)

    def occupancy(t, st):
        peak[0] = max(peak[0], int(st["lane_n"].sum(axis=1).max()))
        peak[1] = max(peak[1], int(((st["flags"] & 1) != 0).sum(axis=1).max()))

    tally, _ = drive([scene], orc, tabs, ticks, seed=11, policy=policy, fill=fill,
                     garbage=opts.get("zero_uncontrolled_actions", False), every_tick=occupancy)
    assert_nontrivial(tally, case)
    assert peak[0] > min_v or peak[1] > min_a, ("no intersection outgrows the next smaller class", case, peak)
    assert scene.stats()["q5_undefined"] == 0


def test_warmup_off_and_collision_threshold_3():
    """No warm-up tick (the reset row is all zeros) and another collision threshold, in a large class."""
    tabs = synthetic_arrivals(4, 1200, 40.0, seed=4, rows=40)
    scene = P.make_scene("emul", 4, vm=5, collision_thr=3, veh_cap=384, agent_cap=320)
    orc = P.make_oracle(4, vm=5, collision_thr=3, veh_cap=scene.veh_cap)
    tally, _ = drive([scene], orc, tabs, 300, seed=4, warmup=False)
    assert_nontrivial(tally, "warmup off")


@GPU
def test_dual_kernel_mode_statistics(monkeypatch):
    """The default launch of the 192/128 class runs two kernels (the intersections that fit the small class, and on a
    second stream the others; PVE_DUAL=0 runs one).  A batch of sparse and dense intersections puts intersections in
    both kernels on every tick after the first 120; both launches must equal the oracle and each other bit for bit."""
    tabs = np.concatenate([synthetic_arrivals(4, 400, 50.0, seed=6, rows=60), synthetic_arrivals(4, 2400, 50.0, seed=7, rows=60)])
    monkeypatch.setenv("PVE_DUAL", "1")
    dual = P.make_scene("cuda", 8, vm=5, veh_cap=192, agent_cap=128)
    monkeypatch.setenv("PVE_DUAL", "0")
    single = P.make_scene("cuda", 8, vm=5, veh_cap=192, agent_cap=128)
    info = dual.launch_info
    assert info["dual"] is True and single.launch_info["dual"] is False
    svc, sac = info["small_veh_cap"], info["small_agent_cap"]
    both = []

    def split(t, st):
        nv, nc = st["lane_n"].sum(axis=1), ((st["flags"] & 1) != 0).sum(axis=1)
        big = (nv > svc) | (nc > sac)                           # cannot fit the small class whatever arrives
        small = (nv + 12 <= svc) & (nc + 12 <= sac)             # fits it even if every lane spawns
        if t >= 120:
            both.append(bool(big.any() and small.any()))

    orc = P.make_oracle(8, vm=5, veh_cap=192)
    tally, (got_dual, got_single) = drive([dual, single], orc, tabs, 320, seed=12, every_tick=split)
    assert len(both) == 200 and all(both)
    assert np.array_equal(env_stats(dual), env_stats(single))
    assert dual.stats() == single.stats()
    assert_nontrivial(tally, "dual")


def test_rows_suppressed_by_out_cap_are_still_counted():
    """out_cap too small for a tick's rows: the intersections whose block does not fit emit no rows (and raise the
    sticky overflow counter), but the statistics describe the simulation, not the emitted rows."""
    _out_cap_case("emul")


@GPU
def test_rows_suppressed_by_out_cap_are_still_counted_cuda():
    _out_cap_case("cuda")


def _out_cap_case(backend):
    B = 8
    tabs = synthetic_arrivals(B, 1000, 40.0, seed=21, rows=32)
    scene = P.make_scene(backend, B, vm=5, out_cap=120)
    orc = P.make_oracle(B, vm=5, veh_cap=scene.veh_cap)
    suppressed = []

    def rows(t, st):
        suppressed.append(int(orc.count_agents()) > 120)

    tally, (got,) = drive([scene], orc, tabs, 300, seed=3, every_tick=rows)
    assert sum(suppressed) > 100
    s = scene.stats()
    assert s["overflow"] > 0 and s["agent_steps"] == tally.s[:, Q["agent_steps"]].sum()
    assert_nontrivial(tally, "out_cap")


# ---- 3. entry points and lifecycle ----------------------------------------------------------------------------------
HOST_MODES = [pytest.param("emul", "staged", id="emul-step_host"),
              pytest.param("cuda", "zerocopy", marks=GPU, id="cuda-step_host_zerocopy"),
              pytest.param("cuda", "staged", marks=GPU, id="cuda-step_host_staged"),
              pytest.param("cuda", "async", marks=GPU, id="cuda-step_host_async")]


@pytest.mark.parametrize("backend,mode", HOST_MODES)
def test_host_entry_points(backend, mode, monkeypatch):
    """``step_host`` (pinned buffers the kernel writes in place, or staged copies with PVE_HOST_ZEROCOPY=0) and the
    pipelined ``step_host_async`` / ``host_wait`` (three ticks in flight): the statistics against the oracle and against
    the rows that reached the host."""
    if mode == "staged":
        monkeypatch.setenv("PVE_HOST_ZEROCOPY", "0")
    B, ticks = 8, 240
    tabs = synthetic_arrivals(B, 1200, 40.0, seed=15, rows=40)
    scene = P.make_scene(backend, B, vm=5)
    orc = P.make_oracle(B, vm=5, veh_cap=scene.veh_cap)
    scene.reset(tabs, warmup=True)
    orc.reset(tabs, warmup=True)
    base = check_reset_row(scene, True)
    ref, rows = Tally(B), Tally(B)
    rng = np.random.RandomState(5)
    pinned = backend == "cuda"
    acts = [torch.zeros(B, scene.veh_cap, dtype=torch.float32) for _ in range(3)]
    if pinned:
        acts = [a.pin_memory() for a in acts]
    pairs = scene.make_async_buffers() if mode == "async" else None
    host = scene.make_host_outputs() if mode != "async" else None
    if mode == "zerocopy":
        assert host.reward.is_pinned() and acts[0].is_pinned()
    pending = []

    def take(n, h, n_veh):
        if mode == "async":
            rec = h.records(n)
            reward, status, cpv, jerk = rec["reward"], rec["status"], rec["cpv"], rec["jerk_sum"]
        else:
            reward, status, cpv, jerk = (getattr(h, f)[:n].numpy() for f in ("reward", "status", "cpv", "jerk_sum"))
        rows.add_rows(h.agent_offset.numpy(), n_veh, cpv, status, jerk, reward, h.env_lock.numpy(),
                      h.env_removed.numpy(), np.zeros(B))

    for t in range(ticks):
        st = orc.get_state()
        a = P.random_actions(rng, (st["flags"] & 1) != 0)
        o = orc.step(a)
        ref.add_oracle(st, o)
        buf = acts[t % 3]                      # the tick that used this buffer last has been waited for
        buf.copy_(torch.from_numpy(a))
        n_veh = st["lane_n"].sum(axis=1)
        if mode == "async":
            scene.step_host_async(buf, pairs[t % 3])
            pending.append((n_veh, len(o["reward"])))
            if t >= 2:
                n, h = scene.host_wait()
                nv, want_n = pending.pop(0)
                assert n == want_n
                take(n, h, nv)
        else:
            n = scene.step_host(buf, host)
            assert n == len(o["reward"])
            take(n, host, n_veh)
    while pending:
        n, h = scene.host_wait()
        nv, want_n = pending.pop(0)
        assert n == want_n
        take(n, h, nv)
    got = env_stats(scene) - base
    compare_stats(got, ref, ORACLE_TOL, "host path, oracle")
    compare_stats(got, rows, ROWS_TOL, "host path, delivered rows", skip=("q5_undefined",))
    P.compare_states(scene.get_state(), orc.get_state(), "host path final")
    check_reduction(scene)
    assert_nontrivial(ref, mode)


@pytest.mark.parametrize("backend", BACKENDS)
def test_statistics_survive_set_state_and_reset_clears_them(backend):
    """Teacher forcing does not touch the statistics: the scene runs 80 ticks of episode A, is then switched by
    ``set_state`` to the state of a second oracle that ran other actions, and follows that one for 160 more ticks; its
    statistics are A's first 80 ticks plus the second oracle's next 160.  A second ``reset`` of the same handle starts a
    new episode from zero."""
    B = 4
    tabs = synthetic_arrivals(B, 1200, 45.0, seed=23, rows=40)
    scene = P.make_scene(backend, B, vm=5)
    oa, ob = P.make_oracle(B, vm=5, veh_cap=scene.veh_cap), P.make_oracle(B, vm=5, veh_cap=scene.veh_cap)
    scene.reset(tabs, warmup=True)
    base = check_reset_row(scene, True)
    tally = Tally(B)
    rng = np.random.RandomState(8)
    for o in (oa, ob):
        o.reset(tabs, warmup=True)
    for t in range(240):
        if t < 80:                                      # episode A on the scene; the second oracle runs its own actions
            st = oa.get_state()
            a = P.random_actions(rng, (st["flags"] & 1) != 0)
            tally.add_oracle(st, oa.step(a))
            ob.step(P.random_actions(rng, ob.control_mask()))
        else:
            st = ob.get_state()
            if t == 80 or t % 40 == 0:                  # switch, then keep forcing now and then (a no-op on the state)
                scene.set_state(P.oracle_state_for_device(st))
                compare_stats(env_stats(scene) - base, tally, ORACLE_TOL, "right after set_state, tick %d" % t)
            a = P.random_actions(rng, (st["flags"] & 1) != 0)
            tally.add_oracle(st, ob.step(a))
        scene.step(P.to_device_actions(scene, a))
        compare_stats(env_stats(scene) - base, tally, ORACLE_TOL, "tick %d" % t)
    P.compare_states(scene.get_state(), ob.get_state(), "after teacher forcing")
    check_reduction(scene)
    assert_nontrivial(tally, "set_state")
    # a new episode on the same handle: other tables, no warm-up this time
    tabs2 = synthetic_arrivals(B, 900, 45.0, seed=24, rows=40)
    orc = P.make_oracle(B, vm=5, veh_cap=scene.veh_cap)
    tally2, _ = drive([scene], orc, tabs2, 120, seed=9, warmup=False)
    s = scene.stats()
    assert s["agent_steps"] == tally2.s[:, Q["agent_steps"]].sum() and s["env_steps"] == B * 120


def q5_state(cap):
    """Two crafted intersections (the builders of crafted.npz's ``q5_ghost_collision``): in 0 an uncontrolled vehicle
    carrying collision > 0 comes first in processing order (lane 0, j = 0), so its -10 has no previous agent to land on
    (the reference's ``reward[-1]`` would raise, the count is ``q5_undefined``); in 1 an agent precedes it and takes the
    -10."""
    rng = np.random.RandomState(20261017)
    ghost = dict(control=False, collision=1, v=10.0)
    s0 = MG.blank_state()
    MG.add_veh(s0, 0, -20.0, **ghost)
    MG.add_veh(s0, 0, 50.0)
    MG.add_veh(s0, 1, 40.0)
    MG.add_veh(s0, 2, -40.0, control=False, collision=3, v=10.0)
    MG.add_veh(s0, 5, 60.0)
    s1 = MG.blank_state()
    MG.add_veh(s1, 0, 90.0)
    MG.add_veh(s1, 1, -20.0, **ghost)
    MG.add_veh(s1, 1, 50.0)
    MG.add_veh(s1, 5, 60.0)
    st = snapshot_to_state(MG.finalize(s0, rng), 2, cap, env=0)
    return snapshot_to_state(MG.finalize(s1, rng), 2, cap, env=1, state=st)


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("caps", [(128, 96), (384, 320)])
def test_q5_undefined_and_the_ghost_reward(backend, caps):
    scene = P.make_scene(backend, 2, vm=5, veh_cap=caps[0], agent_cap=caps[1])
    orc = P.make_oracle(2, vm=5, veh_cap=scene.veh_cap)
    far = np.full((64, 12), 1e6)
    scene.reset(far, warmup=False)
    orc.reset(far, warmup=False)
    base = check_reset_row(scene, False)
    st = q5_state(scene.veh_cap)
    orc.set_state(st)
    scene.set_state(P.oracle_state_for_device(st))
    act = np.zeros((2, scene.veh_cap), np.float32)
    o = orc.step(act)
    out = P.outputs_to_numpy(scene.step(P.to_device_actions(scene, act)))
    P.compare_outputs(out, o, "q5 tick")
    np.testing.assert_array_equal(o["q5_undefined"], [1, 0])
    lo, hi = o["agent_offset"][1], o["agent_offset"][2]
    assert o["reward"][lo] == -10 and out["reward"][lo] == -10         # the agent ahead of the ghost of intersection 1
    tally = Tally(2)
    tally.add_oracle(st, o)
    got = env_stats(scene) - base
    compare_stats(got, tally, ORACLE_TOL, "q5 tick")
    np.testing.assert_array_equal(got[:, Q["q5_undefined"]], [1, 0])
    assert abs(got[1, Q["reward_sum"]] - out["reward"][lo:hi].astype(np.float64).sum()) <= 1e-12 * 20 * (hi - lo)
    s, _, _ = check_reduction(scene)
    assert s["q5_undefined"] == 1 and s["removed"] == got[:, Q["removed"]].sum() >= 3


# ---- 4. the 4- and 8-lane kernel ------------------------------------------------------------------------------------
@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("lanes", [4, 8])
@pytest.mark.parametrize("caps", [None, (64, 64)], ids=["class_128_96", "class_64_64"])
def test_lane4_and_lane8_statistics(backend, lanes, caps, monkeypatch):
    """The one-warp kernel of ``lane_num`` 4 and 8 (csrc/scene_step4.cuh) against its per-intersection Python oracles."""
    from oracle.scene4_oracle import Scene4Oracle
    from oracle.scene8_oracle import Scene8Oracle
    monkeypatch.setattr(E4, "CAPS4", caps)
    B, ticks, seed = 4, 260, 5 + lanes
    tabs = synthetic_arrivals(B, 1400 if lanes == 4 else 1000, ticks * 0.1 + 30.0, seed=seed)[:, :, :lanes].copy()
    scene = E4.make_scene4(backend, B, lanes=lanes)
    assert caps is None or scene.veh_cap == caps[0]
    if lanes == 4:
        scene.reset(tabs, warmup=True)
        orcs = [Scene4Oracle() for _ in range(B)]
        for b, o in enumerate(orcs):
            o.reset(tabs[b], warmup=True)
    else:
        draws = np.random.RandomState(seed + 100).randint(0, 2, size=(B,) + tabs.shape[1:]).astype(np.uint8)
        scene.reset(tabs, warmup=True, intention_draws=draws)
        orcs = [Scene8Oracle() for _ in range(B)]
        for b, o in enumerate(orcs):
            o.reset(tabs[b], draws[b], warmup=True)
    base = check_reset_row(scene, True)
    tally = Tally(B)
    rng = np.random.RandomState(seed)
    for t in range(ticks):
        act = np.zeros((B, scene.veh_cap), np.float32)
        vals = np.zeros((B, len(NAMES)))
        mags = np.zeros((B, len(NAMES)))
        for b, o in enumerate(orcs):
            m = np.array(o.control_mask(), bool)
            act[b, :len(m)] = np.where(m, rng.uniform(-3, 3, size=len(m)), 0.0)
        scene.step(P.to_device_actions(scene, act))
        for b, o in enumerate(orcs):
            V = sum(len(x) for x in o.lanes)
            ref = o.step(act[b, :V])
            r = np.array(ref["reward"], np.float64)
            jk = np.array(ref["jerks"], np.float64)
            vals[b] = [len(ref["ids"]), V, int((np.array(ref["cpv"]) > 0).sum()), ref["lock"], jk.sum(), r.sum(),
                       (r * r).sum(), ref["n_removed"], 1, 0]
            mags[b] = np.abs(vals[b])
            mags[b, Q["passed_jerk_sum"]], mags[b, Q["reward_sum"]] = np.abs(jk).sum(), np.abs(r).sum()
        tally.s += vals
        tally.mag += mags
        compare_stats(env_stats(scene) - base, tally, ORACLE_TOL, "lanes=%d tick %d" % (lanes, t))
    check_reduction(scene)
    assert_nontrivial(tally, "lanes=%d" % lanes)


# ---- 5. the end-of-rollout reduction --------------------------------------------------------------------------------
@pytest.mark.parametrize("backend,B", [("emul", 1), ("emul", 255), ("emul", 257),
                                       pytest.param("cuda", 1, marks=GPU), pytest.param("cuda", 255, marks=GPU),
                                       pytest.param("cuda", 257, marks=GPU), pytest.param("cuda", 5000, marks=GPU)])
def test_end_of_rollout_reduction(backend, B):
    """``pve_stats`` (one 256-thread CTA, a strided loop over the intersections) against the column sums of the
    per-intersection statistics and the header counters, and the statistics against the rows the scene delivered.
    Every 16th intersection is fed a vehicle every 0.5 s on every lane: it outgrows the 128-vehicle class, drops
    arrivals, and the overflow slot is not zero."""
    ticks = 150
    tabs = synthetic_arrivals(B, 1000, 30.0, seed=B, rows=40)
    tabs[::16] = 0.5 * np.arange(1, tabs.shape[1] + 1)[:, None]
    scene = P.make_scene(backend, B, vm=5)
    scene.reset(tabs, warmup=True)
    base = check_reset_row(scene, True)
    tally = Tally(B)
    rng = np.random.RandomState(B)
    for t in range(ticks):
        n_veh = vehicles_now(scene)
        act = P.random_actions(rng, scene.control_mask().cpu().numpy())
        rows_tally(tally, n_veh, scene.step(P.to_device_actions(scene, act)))
    compare_stats(env_stats(scene) - base, tally, ROWS_TOL, "B=%d" % B, skip=("q5_undefined",))
    s, es, st = check_reduction(scene)
    assert s["overflow"] > 0 and s["env_steps"] == B * (ticks + 1) and s["q5_undefined"] == 0
    assert s["spawned"] - s["removed"] == int(st["n_veh"].sum())


# ---- 6. the evaluation report ---------------------------------------------------------------------------------------
@GPU
def test_evaluation_report_equals_the_python_loop_tallies():
    """``evaluate_tables`` (the library's rollout loop, tallies from the per-intersection statistics) against the same
    closed loop driven from Python on a second scene and tallied from the rows as main.py:407-415 does."""
    from pve_mcc_for_unsignalized_intersection_b200 import evaluate
    from pve_mcc_for_unsignalized_intersection_b200.actor import ActorWeights, BatchedActor
    w = ActorWeights.from_npz(os.path.join(P.ROOT, "tests", "golden", "actor_agent1.npz"))
    tables = [synthetic_arrivals(1, 1800, 160.0, seed=41)[0], synthetic_arrivals(1, 1000, 100.0, seed=42)[0],
              synthetic_arrivals(1, 400, 60.0, seed=43)[0]]          # dense, medium, and one that runs dry early
    ticks, caps = 1500, dict(veh_cap=192, agent_cap=128)
    res = evaluate.evaluate_tables(tables, w, ticks=ticks, **caps)
    B = len(tables)
    scene = P.make_scene("cuda", B, vm=5, **caps)
    actor = BatchedActor(w)
    scene.reset(evaluate.stack_tables(tables), warmup=True)
    acts = torch.empty(B, scene.veh_cap, dtype=torch.float32, device="cuda")
    coll = torch.zeros(B, dtype=torch.int64, device="cuda")
    lock = torch.zeros(B, dtype=torch.int64, device="cuda")
    jerk = torch.zeros(B, dtype=torch.float64, device="cuda")
    for _ in range(ticks):
        out = scene.step(actor.act(scene, out=acts))
        n = out.n_agents
        env = out.ids[:n, 0].long()
        coll.index_add_(0, env, (out.cpv[:n] > 0).long())                                   # main.py:410-412
        lock += out.env_lock.long()                                                          # main.py:408
        fin = (out.status[:n] & N.ST_FINISHED) != 0
        jerk.index_add_(0, env, torch.where(fin, out.jerk_sum[:n].double(), torch.zeros_like(jerk[:1])))   # main.py:409
    st = scene.get_state()
    coll, lock, jerk = coll.cpu().numpy(), lock.cpu().numpy(), jerk.cpu().numpy()
    for b, r in enumerate(res):
        want = [int(st["id_seq"][b]), int(coll[b]), int(st["passed_veh"][b]), int(lock[b]), int(st["passed_step_total"][b])]
        assert [r["vehicles"], r["collisions"], r["passed"], r["lock_total"], r["passed_step_total"]] == want, (b, r, want)
        assert abs(r["jerk_total"] - jerk[b]) <= 1e-6 * jerk[b], (b, r["jerk_total"], jerk[b])
        # the jerk tally of the rows is float32 per vehicle: the line is compared with the device's float64 total
        assert r["report"] == evaluate.format_report(want[0], want[1], want[2], want[4], r["jerk_total"], want[3])
    assert res[0]["collisions"] > 0 and all(r["lock_total"] > 0 for r in res)
    assert len({r["vehicles"] for r in res}) == 3
