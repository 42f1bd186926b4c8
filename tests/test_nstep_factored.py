"""GPU tier, row N2 with the factored frame log: ``NStepFolder(factored=True)`` (``pve_nstep_create_factored`` /
``pve_nstep_push_factored``) keeps per push the factored observation (row 0, previous row 0, 8 row codes and the
push's agent offsets) instead of the 7 x 28 blocks, and expands the frames into the replay records.

Its replay memory, counters and bootstrap values must be those of a full-frame folder fed the same ticks, bit for bit,
with every implementation of the two target networks; the folder has no emulation build, so every test needs a GPU.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import nstep_common as K
from oracle import nstep_oracle
from pve_mcc_for_unsignalized_intersection_b200 import SceneConfig
from pve_mcc_for_unsignalized_intersection_b200 import _native as N
from pve_mcc_for_unsignalized_intersection_b200.actor import ActorWeights, BatchedActor
from pve_mcc_for_unsignalized_intersection_b200.arrivals import synthetic_arrivals
from pve_mcc_for_unsignalized_intersection_b200.nstep import BatchedCritic, CriticWeights, NStepFolder
from pve_mcc_for_unsignalized_intersection_b200.scene import BatchedScene, StepOutputs

pytestmark = pytest.mark.gpu

# as tests/test_gpu_nstep.py: float32 rewards summed over <= 13 terms plus gamma^n * Q'
T_RTOL, T_ATOL = 1e-5, 2e-4
RECORD_KEYS = ("state", "action", "reward", "next_state", "done")


def nets():
    a, c = K.load_nets()
    return ActorWeights(a), CriticWeights(c)


def make(B, lane_num=12, **kw):
    return BatchedScene(B, SceneConfig(vm=6, collision_thr=2, lane_num=lane_num), device="cuda:0", **kw)


def full_twin(B):
    """Today's training path: observation blocks, neighbour sources, full-frame folder pushed with push_scene."""
    return make(B, neighbour_sources=True)


def factored_scene(B, full_obs=False):
    return make(B, factored_obs=True, full_obs=full_obs)


def random_actions(gen, scene):
    return ((torch.rand(scene.B, scene.veh_cap, device="cuda", generator=gen) * 6 - 3) * scene.control_mask()).contiguous()


def assert_same_memory(a, b, what=""):
    ca, cb = a.counters(), b.counters()
    assert ca["num_experiences"] == cb["num_experiences"] and ca["last_added"] == cb["last_added"], (what, ca, cb)
    assert ca["slot_conflicts"] == 0 and cb["slot_conflicts"] == 0, (what, ca, cb)
    n = min(ca["num_experiences"], a.capacity)
    for k in RECORD_KEYS:
        x, y = a.arrays()[k][:n], b.arrays()[k][:n]
        if x.dtype == torch.float32:           # bit patterns: NaN rows and signed zeros compare exactly
            x, y = x.contiguous().view(torch.int32), y.contiguous().view(torch.int32)
        assert torch.equal(x, y), (what, k)
    return ca["num_experiences"]


@pytest.mark.parametrize("impl", ["tc5", "mma", "ffma"])
def test_factored_folder_equals_the_full_frame_folder(impl, monkeypatch):
    """B = 512, seq_max_step 12, 220 ticks of U(-3, 3) actions: bootstrap values every 20 ticks and the whole replay
    memory (over a million records) bit for bit, with each implementation of the target actor and critic."""
    monkeypatch.setenv("PVE_ACTOR_IMPL", impl)
    monkeypatch.setenv("PVE_CRITIC_IMPL", impl)
    aw, cw = nets()
    B, S = 512, 12
    tabs = synthetic_arrivals(B, 1000, 40.0, seed=8)
    sa, sb = full_twin(B), factored_scene(B)
    for s in (sa, sb):
        s.reset(tabs, warmup=False)
    actor, critic = BatchedActor(aw), BatchedCritic(cw)
    full = NStepFolder(sa, actor, critic, S, buffer_size=3_000_000)
    fact = NStepFolder(sb, actor, critic, S, buffer_size=3_000_000, factored=True)
    gen = torch.Generator(device="cuda").manual_seed(2)
    for t in range(220):
        acts = random_actions(gen, sa)
        full.bind_outputs()
        oa = sa.step(acts)
        full.push(oa, 0.85)                                      # push_scene: nbr_src of scene.out
        fact.bind_outputs()
        ob = sb.step(acts)
        fact.push(ob, 0.85)
        if t % 20 == 19:
            n = oa.n_agents
            assert n == ob.n_agents
            assert torch.equal(full.bootstrap_values()[:n], fact.bootstrap_values()[:n]), t
    n = assert_same_memory(full, fact, impl)
    assert n > 1_000_000


def test_log_wraps_episode_reset_bound_and_copied():
    """B = 256, seq_max_step 5 (the log wraps every 7 pushes), 150 ticks with a new episode at tick 70: a factored folder
    whose step writes into the log (bind_outputs) and one that copies from scene.out both equal the full-frame twin."""
    aw, cw = nets()
    B, S = 256, 5
    tabs = synthetic_arrivals(B, 1000, 40.0, seed=11)
    twin, bound, copied = full_twin(B), factored_scene(B), factored_scene(B, full_obs=True)
    scenes = (twin, bound, copied)
    for s in scenes:
        s.reset(tabs, warmup=False)
    folders = (NStepFolder(twin, BatchedActor(aw), BatchedCritic(cw), S, buffer_size=1_000_000),
               NStepFolder(bound, BatchedActor(aw), BatchedCritic(cw), S, buffer_size=1_000_000, factored=True),
               NStepFolder(copied, BatchedActor(aw), BatchedCritic(cw), S, buffer_size=1_000_000, factored=True))
    gen = torch.Generator(device="cuda").manual_seed(5)
    for t in range(150):
        acts = random_actions(gen, twin)
        if t == 70:
            for f in folders:
                f.reset()                                        # a new episode: buffers dropped, memory kept
        folders[1].bind_outputs()
        for s, f in zip(scenes, folders):
            f.push(s.step(acts), 0.9)
    n = assert_same_memory(folders[0], folders[1], "bound")
    assert assert_same_memory(folders[0], folders[2], "copied") == n > 100_000


@pytest.mark.parametrize("S", [0, 14])
def test_seq_max_step_edges(S):
    """The smallest and the largest frame log (M = 2 and 16 pushes) against the full-frame twin."""
    aw, cw = nets()
    B = 64
    tabs = synthetic_arrivals(B, 1200, 30.0, seed=S)
    twin, fs = full_twin(B), factored_scene(B)
    for s in (twin, fs):
        s.reset(tabs, warmup=True)
    actor, critic = BatchedActor(aw), BatchedCritic(cw)
    full = NStepFolder(twin, actor, critic, S, buffer_size=200_000)
    fact = NStepFolder(fs, actor, critic, S, buffer_size=200_000, factored=True)
    gen = torch.Generator(device="cuda").manual_seed(S + 1)
    for t in range(60):
        acts = random_actions(gen, twin)
        full.push(twin.step(acts), 0.5)
        fact.bind_outputs()
        fact.push(fs.step(acts), 0.5)
    assert assert_same_memory(full, fact, S) > 0


def test_against_the_oracle():
    """Two episodes on the same tables; the oracle is fed the factored outputs expanded with expand_obs(): states
    exactly, targets within the n-step bound."""
    aw, cw = nets()
    B, S = 6, 5
    tabs = synthetic_arrivals(B, 1000, 30.0, seed=21)
    scene = factored_scene(B)
    folder = NStepFolder(scene, BatchedActor(aw), BatchedCritic(cw), S, buffer_size=100000, factored=True)
    orc = nstep_oracle.NStepOracle(aw, cw, S, buffer_size=100000)
    gen = torch.Generator(device="cuda").manual_seed(9)
    n_prev = 0
    for episode in range(2):
        scene.reset(tabs, warmup=True)
        folder.reset()
        orc.reset()
        for t in range(70):
            folder.bind_outputs()
            out = scene.step(random_actions(gen, scene))
            obs = out.expand_obs().cpu().numpy()                # before the push: the next bind moves the outputs
            n = out.n_agents
            ids, reward = out.ids[:n].cpu().numpy(), out.reward[:n].cpu().numpy()
            done = (out.status[:n].cpu().numpy() & K.ST_DONE) != 0
            folder.push(out, 0.7)
            added = orc.push(ids[:, 0], ids[:, 3], obs, reward, done, 0.7)
            c = folder.counters()
            assert c["num_experiences"] == n_prev + len(added), (episode, t)
            idx = torch.arange(n_prev, c["num_experiences"], device="cuda") % folder.capacity
            rec = {k: v.index_select(0, idx).cpu().numpy() for k, v in folder.arrays().items()}
            for i, (row, state, action, target, nxt) in enumerate(added):
                assert np.array_equal(rec["state"][i], state.astype(np.float32)), (episode, t, i)
                assert np.array_equal(rec["next_state"][i], nxt.astype(np.float32)), (episode, t, i)
                assert np.array_equal(rec["action"][i], action.astype(np.float32)), (episode, t, i)
                assert abs(rec["reward"][i] - target) <= T_RTOL * abs(target) + T_ATOL, (episode, t, i)
            n_prev = c["num_experiences"]
    assert n_prev > 1000 and folder.counters()["slot_conflicts"] == 0


def test_a_push_may_lag_the_step():
    """Tick t is pushed after step t + 1 has run, from one of three rotating device outputs: the memory equals that of
    a folder that pushes every tick at once."""
    aw, cw = nets()
    B, S = 256, 12
    tabs = synthetic_arrivals(B, 1000, 40.0, seed=4)
    now, late = factored_scene(B), factored_scene(B)
    for s in (now, late):
        s.reset(tabs, warmup=False)
    actor, critic = BatchedActor(aw), BatchedCritic(cw)
    f_now = NStepFolder(now, actor, critic, S, buffer_size=1_000_000, factored=True)
    f_late = NStepFolder(late, actor, critic, S, buffer_size=1_000_000, factored=True)
    outs = [StepOutputs(B, late.out_cap, late.device, factored=True, full_obs=False, lib=late.lib) for _ in range(3)]
    natives = [o.native() for o in outs]
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    gen = torch.Generator(device="cuda").manual_seed(6)
    ticks = 120
    for t in range(ticks):
        acts = random_actions(gen, now)
        f_now.bind_outputs()
        f_now.push(now.step(acts), 0.9)
        late._check(late.lib.pve_step(late._h, acts.data_ptr(), C.byref(natives[t % 3]), stream))
        if t >= 1:
            f_late.push(outs[(t - 1) % 3], 0.9)                # step t has already run
    f_late.push(outs[(ticks - 1) % 3], 0.9)
    assert assert_same_memory(f_now, f_late, "lagged") > 100_000


def test_at_size_and_the_log_is_smaller():
    """BASELINE config 2 size (4 096 intersections), 80 ticks after 150 priming ticks: records equal to the full-frame
    twin, bit for bit; the factored frame log takes at most 0.31 of the full-frame log."""
    aw, cw = nets()
    B, S = 4096, 12
    tabs = synthetic_arrivals(B, 1000, 40.0, seed=3)
    twin, fs = full_twin(B), factored_scene(B)
    gen = torch.Generator(device="cuda").manual_seed(7)
    for s in (twin, fs):
        s.reset(tabs, warmup=False)
    for _ in range(150):
        acts = random_actions(gen, twin)
        twin.step(acts)
        fs.step(acts)
    actor, critic = BatchedActor(aw), BatchedCritic(cw)
    full = NStepFolder(twin, actor, critic, S, buffer_size=4_000_000)
    fact = NStepFolder(fs, actor, critic, S, buffer_size=4_000_000, factored=True)
    assert full.log_bytes == (S + 2) * twin.out_cap * 7 * 28 * 4
    assert fact.log_bytes == (S + 2) * (fs.out_cap * (2 * 28 * 4 + 8 * 2) + (B + 1) * 4)
    assert fact.log_bytes <= 0.31 * full.log_bytes
    for t in range(80):
        acts = random_actions(gen, twin)
        full.bind_outputs()
        full.push(twin.step(acts), 0.9)
        fact.bind_outputs()
        fact.push(fs.step(acts), 0.9)
    assert assert_same_memory(full, fact, "B=4096") > 1_000_000


def test_refusals():
    aw, cw = nets()
    B = 4
    sa, sb = full_twin(B), factored_scene(B)
    tabs = synthetic_arrivals(B, 1000, 20.0, seed=1, rows=16)
    for s in (sa, sb):
        s.reset(tabs, warmup=True)
    actor, critic = BatchedActor(aw), BatchedCritic(cw)
    full = NStepFolder(sa, actor, critic, 3, buffer_size=10_000)
    fact = NStepFolder(sb, actor, critic, 3, buffer_size=10_000, factored=True)
    acts = torch.zeros(B, sa.veh_cap, device="cuda")
    oa, ob = sa.step(acts), sb.step(acts)
    lib, st = sa.lib, C.c_void_p(torch.cuda.current_stream().cuda_stream)
    both = StepOutputs(B, sa.out_cap, sa.device, neighbour_sources=True, factored=True, lib=lib)   # every field set
    nets_ = (actor._h, critic._h, st)
    # a push that does not match the folder's frame log
    assert lib.pve_nstep_push(fact._h, C.byref(both.native()), 0.9, *nets_) == -1
    assert b"pve_nstep_push_factored" in lib.pve_nstep_last_error(fact._h)
    assert lib.pve_nstep_push_scene(fact._h, sb._h, C.byref(both.native()), 0.9, *nets_) == -1
    assert lib.pve_nstep_push_factored(full._h, C.byref(both.native()), 0.9, *nets_) == -1
    assert b"pve_nstep_create_factored" in lib.pve_nstep_last_error(full._h)
    # a factored push with one of the three fields missing
    for name in ("row0_out", "prev_row0", "obs_src"):
        o = both.native()
        setattr(o, name, None)
        assert lib.pve_nstep_push_factored(fact._h, C.byref(o), 0.9, *nets_) == -1, name
        assert b"row0_out, prev_row0 and obs_src" in lib.pve_nstep_last_error(fact._h)
    # the log slot of the other format
    p = C.c_void_p()
    assert lib.pve_nstep_obs_slot(fact._h, C.byref(p)) == -4
    assert lib.pve_nstep_factored_slot(full._h, C.byref(C.c_void_p()), C.byref(C.c_void_p()), C.byref(C.c_void_p())) == -4
    # nothing above reached the device: both folders still take their own pushes
    assert fact.counters()["pushes"] == 0 and full.counters()["pushes"] == 0
    full.push(oa, 0.9)
    fact.push(ob, 0.9)
    assert fact.counters()["pushes"] == 1 and full.counters()["pushes"] == 1
    # Python: outputs without the factored fields, scenes that do not export them
    with pytest.raises(ValueError, match="factored_obs=True"):
        fact.push(oa, 0.9)
    with pytest.raises(ValueError, match="factored_obs=True"):
        NStepFolder(sa, actor, critic, 3, buffer_size=10_000, factored=True)
    s4 = make(B, lane_num=4)
    with pytest.raises(ValueError, match="factored_obs=True"):
        NStepFolder(s4, actor, critic, 3, buffer_size=10_000, factored=True)
