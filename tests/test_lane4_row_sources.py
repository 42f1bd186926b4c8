"""Row sources (``pve_outputs.nbr_src``) of the 4- and 8-lane step (csrc/scene_step4.cuh, ``SRC`` instantiation) and the
distinct-row bootstrap of the n-step folder (``pve_nstep_push_scene``) on those geometries.

CPU tier: the kernel source compiled as the sequential emulation.  GPU tier (``gpu`` marker): the CUDA build in both
capacity classes, at 4 096 intersections, and the folder fed by ``push`` against ``push_scene``."""
import numpy as np
import pytest
import torch

from pve_mcc_for_unsignalized_intersection_b200 import SceneConfig
from pve_mcc_for_unsignalized_intersection_b200.arrivals import synthetic_arrivals
from pve_mcc_for_unsignalized_intersection_b200.scene import BatchedScene

OUT_FIELDS = ("agent_offset", "obs", "reward", "ids", "cpv", "status", "jerk_sum", "env_collisions", "env_lock", "env_removed")


def make_scene(backend, B, lanes, caps=(128, 96), src=True, vm=5):
    cfg = SceneConfig(vm=vm, collision_thr=2, lane_num=lanes)
    kw = dict(veh_cap=caps[0], agent_cap=caps[1], neighbour_sources=src)
    if backend == "cuda":
        return BatchedScene(B, cfg, device="cuda:0", **kw)
    from emul.build_emul import build_emul
    return BatchedScene(B, cfg, device="cpu", _library=build_emul(), **kw)


def reset(scene, lanes, arrivals, density, seed, seconds):
    if arrivals == "poisson":
        scene.reset_poisson(density, seed)
        return
    B = scene.B
    tabs = synthetic_arrivals(B, density, seconds, seed=seed)[:, :, :lanes].copy()
    draws = np.random.RandomState(seed + 100).randint(0, 2, size=(B, tabs.shape[1], 8)).astype(np.uint8) if lanes == 8 else None
    scene.reset(tabs, warmup=True, intention_draws=draws)


def bits(t):
    a = t.detach().cpu().numpy()
    return a.view(np.int32) if a.dtype == np.float32 else a


def outputs_bits(out):
    n = out.n_agents
    return {f: bits(getattr(out, f)[:n] if f not in ("agent_offset", "env_collisions", "env_lock", "env_removed")
                    else getattr(out, f)) for f in OUT_FIELDS}


def assert_same_outputs(a, b, what):
    for f in OUT_FIELDS:
        np.testing.assert_array_equal(a[f], b[f], err_msg="%s: %s" % (what, f))


def assert_same_state(sa, sb, what):
    """Every field of get_state bit for bit; the stored rows in the slots that hold a vehicle (the slots past n_veh hold
    none, and a step that writes nbr_src leaves other leftovers there than one that does not)."""
    for k in sa:
        if k == "row0":
            continue
        np.testing.assert_array_equal(sa[k], sb[k], err_msg="%s: state %s" % (what, k))
    live = np.arange(sa["row0"].shape[1])[None, :] < sa["n_veh"][:, None]
    np.testing.assert_array_equal(sa["row0"].view(np.int32)[live], sb["row0"].view(np.int32)[live], err_msg=what + ": row0")


def check_codes(out, prev, lane_n, what, seen):
    """Every observation row is bit for bit the row its code names; entry 0 is the row itself, entry 7 is -1, every new
    code names an agent of the intersection and every 0x4000 code the slot of a vehicle that is an agent this tick.
    ``prev``: the stored rows before the step (int32 view), ``lane_n``: the lane counts before the step."""
    n = out.n_agents
    obs = bits(out.obs[:n])
    src = out.nbr_src[:n].cpu().numpy().astype(np.int32)
    ids = out.ids[:n].cpu().numpy()
    off = out.agent_offset.cpu().numpy().astype(np.int64)
    b = ids[:, 0].astype(np.int64)
    r = np.arange(n)
    np.testing.assert_array_equal(src[:, 0], r - off[b], err_msg=what + ": entry 0")
    assert np.all(src[:, 7] == -1), what
    lane_off = np.concatenate([np.zeros((lane_n.shape[0], 1), np.int64), np.cumsum(lane_n, axis=1)], axis=1)
    agent_slot = np.zeros(prev.shape[:2], bool)
    agent_slot[b, lane_off[b, ids[:, 1]] + ids[:, 2]] = True
    for k in range(1, 7):
        v = src[:, k]
        zero, old = v < 0, (v >= 0) & ((v & 0x4000) != 0)
        new = (v >= 0) & ~old
        assert np.all(obs[zero, k] == 0), (what, k)
        assert np.all(off[b[new]] + v[new] < off[b[new] + 1]), (what, k)
        np.testing.assert_array_equal(obs[new, k], obs[off[b[new]] + v[new], 0], err_msg="%s row %d new" % (what, k))
        slot = v[old] & 0x3FFF
        assert np.all(agent_slot[b[old], slot]), (what, k, "0x4000 code names a slot without an agent")
        np.testing.assert_array_equal(obs[old, k], prev[b[old], slot], err_msg="%s row %d prev" % (what, k))
        seen["zero"] += int(zero.sum()); seen["new"] += int(new.sum()); seen["prev"] += int(old.sum())
    seen["left"] += int((np.asarray(out.obs[:n, 0, 3].cpu()).astype(np.int64) % 3 == 0).sum())     # route % 3 == 0 agents


def run_row_sources(backend, lanes, arrivals, B=3, ticks=160, caps=(128, 96), density=1400, seed=5, state_every=10):
    """Three scenes on the same traffic and actions: ``src`` writes nbr_src every tick, ``alt`` every other tick (and
    is teacher-forced with its own state half-way), ``plain`` never.  All three must agree bit for bit."""
    scenes = {k: make_scene(backend, B, lanes, caps, src=(k != "plain")) for k in ("src", "alt", "plain")}
    for s in scenes.values():
        reset(s, lanes, arrivals, density, seed, ticks * 0.1 + 30.0)
    src, alt, plain = scenes["src"], scenes["alt"], scenes["plain"]
    rng = np.random.RandomState(seed)
    seen = {"zero": 0, "new": 0, "prev": 0, "left": 0}
    coll = 0
    for t in range(ticks):
        ctrl = src.control_mask().cpu().numpy()
        act = torch.from_numpy(np.where(ctrl, rng.uniform(-3, 3, size=ctrl.shape), 0).astype(np.float32)).to(src.device)
        if t == ticks // 2:
            for s in (src, alt):
                s.set_state(s.get_state())
        lane_n = src.get_state()["lane_n"][:, :lanes].astype(np.int64)
        prev = bits(src.row0()).copy()
        np.testing.assert_array_equal(bits(alt.row0())[lane_n.sum(1)[:, None] > np.arange(prev.shape[1])[None, :]],
                                      prev[lane_n.sum(1)[:, None] > np.arange(prev.shape[1])[None, :]], err_msg="alt rows")
        o_src = src.step(act)
        check_codes(o_src, prev, lane_n, "%d lanes %s tick %d" % (lanes, arrivals, t), seen)
        # the rows this step read stay readable until the next step
        np.testing.assert_array_equal(bits(src.row0_prev()), prev, err_msg="row0_prev tick %d" % t)
        a_src = outputs_bits(o_src)
        if t % 2:
            alt._out_native.nbr_src = None                  # this tick without nbr_src: the plain instantiation
        try:
            a_alt = outputs_bits(alt.step(act))
        finally:
            alt._out_native = alt.out.native()
        a_plain = outputs_bits(plain.step(act))
        assert_same_outputs(a_src, a_plain, "src/plain tick %d" % t)
        assert_same_outputs(a_alt, a_plain, "alt/plain tick %d" % t)
        coll += int(a_plain["env_collisions"].sum())
        if t % state_every == 0 or t == ticks - 1:
            sp = plain.get_state()
            assert_same_state(src.get_state(), sp, "src tick %d" % t)
            assert_same_state(alt.get_state(), sp, "alt tick %d" % t)
            for s in (src, alt):
                np.testing.assert_array_equal(s.env_stats().cpu().numpy(), plain.env_stats().cpu().numpy())
    assert src.stats() == plain.stats() == alt.stats()
    assert coll > 0 and min(seen.values()) > 20, (coll, seen)
    return seen


# ---- CPU tier --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("arrivals", ["table", "poisson"])
@pytest.mark.parametrize("lanes", [4, 8])
def test_row_sources_name_the_copied_rows(lanes, arrivals):
    run_row_sources("emul", lanes, arrivals, caps=(128, 96) if arrivals == "table" else (64, 64))


def test_lane4_left_turn_rewrite_is_covered():
    """lane_num = 4: agents of the left-turn routes (route % 3 == 0) rewrite the list the agents after them read."""
    seen = run_row_sources("emul", 4, "table", B=2, ticks=120, density=1600, seed=9)
    assert seen["left"] > 200, seen


def test_push_scene_rows_stay_until_the_next_step():
    """row0_prev after a step with nbr_src is the stored rows that step read, also after a step without it (the phase
    only moves with nbr_src: the buffer row0() returns is the same one)."""
    scene = make_scene("emul", 2, 4)
    reset(scene, 4, "table", 1400, 3, 60.0)
    act = torch.zeros(2, scene.veh_cap)
    for _ in range(40):
        scene.step(act)
    before = bits(scene.row0()).copy()
    scene.step(act)
    np.testing.assert_array_equal(bits(scene.row0_prev()), before)
    scene._out_native.nbr_src = None
    try:
        p0 = scene.lib.pve_row0_dev(scene._h)
        scene.step(act)
        assert scene.lib.pve_row0_dev(scene._h) == p0
    finally:
        scene._out_native = scene.out.native()


# ---- GPU tier --------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("caps", [(64, 64), (128, 96)])
@pytest.mark.parametrize("arrivals", ["table", "poisson"])
@pytest.mark.parametrize("lanes", [4, 8])
def test_device_row_sources(lanes, arrivals, caps):
    scene = make_scene("cuda", 1, lanes, caps)
    assert scene.backend == "cuda-sm_100a" and scene.veh_cap == caps[0]
    run_row_sources("cuda", lanes, arrivals, B=8, caps=caps, density=1400 if caps[0] == 128 else 1000)


@pytest.mark.gpu
@pytest.mark.parametrize("lanes", [4, 8])
def test_device_codes_equal_emulation_codes(lanes):
    B, ticks = 4, 120
    dev, emu = make_scene("cuda", B, lanes), make_scene("emul", B, lanes)
    for s in (dev, emu):
        reset(s, lanes, "table", 1200, 7, 60.0)
    rng = np.random.RandomState(1)
    for t in range(ticks):
        ctrl = emu.control_mask().numpy()
        act = np.where(ctrl, rng.uniform(-3, 3, size=ctrl.shape), 0).astype(np.float32)
        od, oe = dev.step(torch.from_numpy(act).cuda()), emu.step(torch.from_numpy(act))
        n = oe.n_agents
        assert od.n_agents == n, t
        np.testing.assert_array_equal(od.nbr_src[:n].cpu().numpy(), oe.nbr_src[:n].numpy(), err_msg="tick %d" % t)
        np.testing.assert_array_equal(od.ids[:n].cpu().numpy(), oe.ids[:n].numpy(), err_msg="tick %d" % t)


@pytest.mark.gpu
@pytest.mark.parametrize("lanes", [4, 8])
def test_device_row_sources_4096(lanes):
    run_row_sources("cuda", lanes, "poisson", B=4096, ticks=100, caps=(64, 64) if lanes == 4 else (128, 96),
                    density=1000, state_every=25)


# ---- the distinct-row bootstrap --------------------------------------------------------------------------------------
def _nets():
    import nstep_common as K
    from pve_mcc_for_unsignalized_intersection_b200.actor import ActorWeights
    from pve_mcc_for_unsignalized_intersection_b200.nstep import CriticWeights
    a, c = K.load_nets()
    return ActorWeights(a), CriticWeights(c)


def run_push_twins(lanes, S, B=256, ticks=200, buffer_size=400_000, reset_at=None, oracle=False, exact=True):
    """Twin scenes, one with nbr_src feeding push_scene, one without feeding push (7 rows per observation): replay
    memory, counters and bootstrap values bit for bit when both pushes run the same network kernels (``exact``: the
    caller pins PVE_ACTOR_IMPL / PVE_CRITIC_IMPL).  Without that, each network call picks its kernel by its own row
    count (mma.sync below 16 384 rows, tcgen05 from there; the zero row's action is computed once, on one row), so the
    7-row and the distinct-row push may run different kernels: then records and counters must still be equal and the
    targets and bootstrap values agree to the networks' tolerance."""
    from oracle import nstep_oracle
    from pve_mcc_for_unsignalized_intersection_b200.actor import BatchedActor
    from pve_mcc_for_unsignalized_intersection_b200.nstep import BatchedCritic, NStepFolder
    aw, cw = _nets()
    actor, critic = BatchedActor(aw), BatchedCritic(cw)
    fast_s, plain_s = make_scene("cuda", B, lanes, vm=6), make_scene("cuda", B, lanes, src=False, vm=6)
    for s in (fast_s, plain_s):
        reset(s, lanes, "table", 1200, 8, ticks * 0.1 + 30.0)
    fast = NStepFolder(fast_s, actor, critic, S, buffer_size=buffer_size)
    plain = NStepFolder(plain_s, actor, critic, S, buffer_size=buffer_size)
    orc = nstep_oracle.NStepOracle(aw, cw, S, buffer_size=buffer_size) if oracle else None
    gen = torch.Generator(device="cuda").manual_seed(2)
    n_prev = 0
    for t in range(ticks):
        if t == reset_at:
            fast.reset(); plain.reset()
            if orc is not None:
                orc.reset()
        acts = ((torch.rand(B, fast_s.veh_cap, device="cuda", generator=gen) * 6 - 3) * fast_s.control_mask()).contiguous()
        of, op = fast_s.step(acts), plain_s.step(acts)
        fast.push(of, 0.85)
        plain.push(op, 0.85, distinct_rows=False)
        n = of.n_agents
        qf, qp = fast.bootstrap_values()[:n], plain.bootstrap_values()[:n]
        if exact:
            assert torch.equal(qf, qp), t
        else:
            assert torch.all((qf - qp).abs() <= Q_RTOL * qp.abs() + Q_ATOL), (t, float((qf - qp).abs().max()))
        if orc is not None:
            ids, obs = of.ids[:n].cpu().numpy(), of.obs[:n].cpu().numpy()
            added = orc.push(ids[:, 0], ids[:, 3], obs, of.reward[:n].cpu().numpy(), (of.status[:n].cpu().numpy() & 1) != 0, 0.85)
            c = fast.counters()
            assert c["num_experiences"] == n_prev + len(added), (t, c, len(added))
            idx = torch.arange(n_prev, c["num_experiences"], device="cuda") % fast.capacity
            rec = {k: v.index_select(0, idx).cpu().numpy() for k, v in fast.arrays().items()}
            for i, (row, state, action, target, nxt) in enumerate(added):
                assert np.array_equal(rec["state"][i], state.astype(np.float32)), (t, i)
                assert np.array_equal(rec["next_state"][i], nxt.astype(np.float32)), (t, i)
                assert abs(rec["reward"][i] - target) <= 1e-5 * abs(target) + 2e-4, (t, i, rec["reward"][i], target)
            n_prev = c["num_experiences"]
    c0, c1 = plain.counters(), fast.counters()
    assert c0 == c1 and c1["slot_conflicts"] == 0 and c1["num_experiences"] > 0, (c0, c1)
    for k in ("state", "action", "next_state"):
        assert torch.equal(plain.arrays()[k], fast.arrays()[k]), k
    rf, rp = fast.arrays()["reward"], plain.arrays()["reward"]
    if exact:
        assert torch.equal(rf, rp)
    else:
        assert torch.all((rf - rp).abs() <= T_RTOL * rp.abs() + T_ATOL), float((rf - rp).abs().max())
    return c1


# two network kernels against each other: tests/test_gpu_nstep.py holds each to 5e-4 of float64 on every row, so they
# may differ by twice that; a target differs by gamma^n times its Q' difference
Q_RTOL, Q_ATOL = 2e-5, 1e-3
T_RTOL, T_ATOL = 2e-5, 1e-3


@pytest.mark.gpu
@pytest.mark.parametrize("impl", ["tc5", "mma", "ffma"])
@pytest.mark.parametrize("lanes", [4, 8])
def test_distinct_row_push_equals_seven_row_push(lanes, impl, monkeypatch):
    monkeypatch.setenv("PVE_ACTOR_IMPL", impl)
    monkeypatch.setenv("PVE_CRITIC_IMPL", impl)
    c = run_push_twins(lanes, 12, buffer_size=100_000, reset_at=120)
    assert c["num_experiences"] > 100_000            # the replay memory wrapped


@pytest.mark.gpu
@pytest.mark.parametrize("S", [0, 14])
@pytest.mark.parametrize("lanes", [4, 8])
def test_distinct_row_push_seq_max_step_edges(lanes, S, monkeypatch):
    monkeypatch.setenv("PVE_ACTOR_IMPL", "tc5")
    monkeypatch.setenv("PVE_CRITIC_IMPL", "tc5")
    run_push_twins(lanes, S, B=64, ticks=120)


@pytest.mark.gpu
@pytest.mark.parametrize("lanes", [4, 8])
def test_distinct_row_push_with_kernels_chosen_by_size(lanes, monkeypatch):
    """The default choice of network kernels: at 64 intersections the 7-row push evaluates 43 008 rows on tcgen05 while
    the distinct-row push evaluates its smaller calls on mma.sync.  Same records, targets within the networks' bounds."""
    monkeypatch.delenv("PVE_ACTOR_IMPL", raising=False)
    monkeypatch.delenv("PVE_CRITIC_IMPL", raising=False)
    run_push_twins(lanes, 0, B=64, ticks=120, exact=False)


@pytest.mark.gpu
@pytest.mark.parametrize("lanes", [4, 8])
def test_distinct_row_push_against_the_oracle(lanes, monkeypatch):
    monkeypatch.setenv("PVE_ACTOR_IMPL", "mma")
    monkeypatch.setenv("PVE_CRITIC_IMPL", "mma")
    run_push_twins(lanes, 6, B=16, ticks=150, buffer_size=20_000, oracle=True)
