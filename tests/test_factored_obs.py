"""The factored observation (``pve_outputs.row0_out`` / ``prev_row0`` / ``obs_src``) and its two expanders.

Every observation row is a copy (Q3): row 0 is the agent's own new row, rows 1-6 are whole stored rows of neighbours,
this tick's or last tick's, or zeros.  A step asked for the factored form writes per agent its row 0, the row stored for
its vehicle when the tick started and 8 row codes; ``expand_obs`` must rebuild ``obs`` from them bit for bit.

Each test runs on the sequential emulation of the kernel source (CPU tier) and, marked ``gpu``, on the CUDA build; the
launch modes that exist on the device only (CTA sizes, the dual-kernel launch, the pipelined host path, the device
expander) run on the GPU only.
"""
import numpy as np
import pytest
import torch

import parity as P
from pve_mcc_for_unsignalized_intersection_b200 import SceneConfig
from pve_mcc_for_unsignalized_intersection_b200 import _native as N
from pve_mcc_for_unsignalized_intersection_b200.arrivals import stress_arrivals, synthetic_arrivals
from pve_mcc_for_unsignalized_intersection_b200.scene import BatchedScene, StepOutputs

GPU = pytest.mark.gpu
BACKENDS = ["emul", pytest.param("cuda", marks=GPU)]
PREV = 0x4000


def make(backend, B, vm=5, veh_cap=128, agent_cap=96, threads=0, out_cap=None, lane_num=12, **kw):
    cfg = SceneConfig(vm=vm, lane_num=lane_num)
    if backend == "cuda":
        return BatchedScene(B, cfg, veh_cap=veh_cap, agent_cap=agent_cap, out_cap=out_cap, device="cuda:0",
                            threads=threads, **kw)
    from emul.build_emul import build_emul
    return BatchedScene(B, cfg, veh_cap=veh_cap, agent_cap=agent_cap, out_cap=out_cap, device="cpu",
                        _library=build_emul(), **kw)


def bits(t):
    """float32 tensor -> its bit patterns (signed zeros and NaN payloads compare exactly)."""
    return t.contiguous().view(torch.int32)


def assert_bits_equal(a, b, what):
    if not torch.equal(bits(a), bits(b)):
        d = (bits(a) != bits(b)).nonzero()
        raise AssertionError("%s: %d values differ, first at %s: %r vs %r" % (
            what, len(d), tuple(d[0].tolist()), a[tuple(d[0])].item(), b[tuple(d[0])].item()))


def header(scene):
    """(lane_n [B, 12] int64, id_seq [B] int64) of the device header, read now."""
    h = scene._wrap(scene.lib.pve_hdr_dev(scene._h), (scene.B, N.HDR_DTYPE.itemsize), torch.uint8, "|u1").clone()
    o = N.HDR_DTYPE.fields["lane_n"][1]
    lane_n = h[:, o:o + 12].to(torch.int64)
    o = N.HDR_DTYPE.fields["id_seq"][1]
    id_seq = h[:, o:o + 4].contiguous().view(torch.int32)[:, 0].to(torch.int64)
    return lane_n, id_seq


def before_step(scene):
    """What a step's factored block is checked against: the stored rows and the header when the tick starts."""
    lane_n, id_seq = header(scene)
    return {"row0": scene.row0().clone(), "lane_n": lane_n, "id_seq": id_seq}


class Checker:
    """Per-tick checks of a scene's factored block; ``prev`` carries the last tick's rows for the uid continuity."""

    def __init__(self):
        self.prev = None
        self.ticks = 0
        self.prev_coded = 0

    def __call__(self, out, pre, n, continuity=True, what=""):
        dev = out.obs_src.device
        off = out.agent_offset.to(torch.int64)
        B = len(off) - 1
        A = off[1:] - off[:-1]
        env = torch.repeat_interleave(torch.arange(B, device=dev), A)
        g = torch.arange(n, device=dev) - off[:-1][env]
        src = out.obs_src[:n].to(torch.int64)
        assert torch.equal(src[:, 0], g), what + ": entry 0 is not the agent itself"
        assert bool((src[:, 7] == -1).all()), what + ": entry 7 is not -1"
        c = src[:, :7]
        valid = (c == -1) | ((c >= 0) & ((c & 0x3FFF) < A[env][:, None]))
        assert bool(valid.all()), what + ": code out of range"
        self.prev_coded += int(((c >= 0) & ((c & PREV) != 0)).sum())
        # the expansion is the observation, bit for bit
        assert_bits_equal(out.expand_obs(n), out.obs[:n], what + ": expand_obs != obs")
        # prev_row0 = the row stored for the agent's slot when the tick started
        lane, j = out.ids[:n, 1].to(torch.int64), out.ids[:n, 2].to(torch.int64)
        start = torch.cumsum(pre["lane_n"], dim=1) - pre["lane_n"]
        slot = start[env, lane] + j
        assert_bits_equal(out.prev_row0[:n], pre["row0"][env, slot], what + ": prev_row0 != stored row of the slot")
        assert_bits_equal(out.row0_out[:n], out.obs[:n, 0], what + ": row0_out != obs[:, 0]")
        # ... = the same vehicle's row0_out of the previous tick, zeros for the vehicles that spawned last tick
        key = (env.cpu().numpy().astype(np.int64) << 32) + out.ids[:n, 3].cpu().numpy().astype(np.int64)
        prev_rows = out.prev_row0[:n].cpu().numpy().view(np.int32)
        if continuity and self.prev is not None:
            pkey, prow, pseq = self.prev
            order = np.argsort(pkey)
            pos = np.searchsorted(pkey[order], key)
            found = (pos < len(pkey)) & (pkey[order][np.minimum(pos, len(pkey) - 1)] == key)
            want = np.zeros_like(prev_rows)
            want[found] = prow[order][pos[found]]
            np.testing.assert_array_equal(prev_rows, want, err_msg=what + ": prev_row0 != last tick's row0_out")
            spawned = (pre["id_seq"] - pseq).cpu().numpy()
            new = np.bincount(env.cpu().numpy()[~found], minlength=B)
            np.testing.assert_array_equal(new, spawned, err_msg=what + ": agents without a row last tick != spawns")
        self.prev = (key, out.row0_out[:n].cpu().numpy().view(np.int32).copy(), pre["id_seq"])
        self.ticks += 1


def mixed_tables(B, rate, seed, rows=48):
    return synthetic_arrivals(B, rate, 45.0, seed=seed, rows=rows)


def actions_for(scene, rng, policy, t, fill):
    ctrl = scene.control_mask().cpu().numpy()
    if policy == "uniform" or (policy == "mixed" and t >= fill and t % 2):
        a = P.random_actions(rng, ctrl)
    else:
        a = np.where(ctrl, -3.0, 0.0).astype(np.float32)
    return P.to_device_actions(scene, a)


# name: (tables, ticks, policy, fill, scene options, gpu only)
CASES = {
    "class_128_80": (lambda: mixed_tables(4, 1400, 3), 300, "uniform", 0, dict(veh_cap=128, agent_cap=80), False),
    "class_128_96": (lambda: mixed_tables(4, 1200, 4), 300, "uniform", 0, dict(veh_cap=128, agent_cap=96), False),
    "class_192_128": (lambda: mixed_tables(4, 2000, 5, rows=60), 300, "uniform", 0, dict(veh_cap=192, agent_cap=128),
                      False),
    "class_384_320_stress": (lambda: stress_arrivals(2, 40.0), 300, "mixed", 200, dict(veh_cap=384, agent_cap=320),
                             False),
    "class_576_416_threads_512": (lambda: stress_arrivals(1, 60.0, headway=0.7), 420, "mixed", 300,
                                  dict(veh_cap=576, agent_cap=416, threads=512), True),
    "dual_4096": (lambda: synthetic_arrivals(4096, 1000, 60.0, seed=17), 160, "uniform", 0, dict(), True),
}
for _nt in (64, 96, 128, 256, 512):        # single-kernel launches of the default class (64, 96: no team / mover split)
    CASES["threads_%d" % _nt] = (lambda: mixed_tables(8, 1400, 8), 300, "uniform", 0, dict(threads=_nt), True)


def _case_params():
    out = []
    for name, case in CASES.items():
        if not case[-1]:
            out.append(pytest.param("emul", name, id="emul-" + name))
        out.append(pytest.param("cuda", name, marks=GPU, id="cuda-" + name))
    return out


@pytest.mark.parametrize("backend,case", _case_params())
def test_expansion_is_the_observation(backend, case):
    """Free-running batches: every tick the factored block expands to ``obs`` bit for bit, ``prev_row0`` is the row
    stored for the agent's slot when the tick started and the same vehicle's ``row0_out`` of the previous tick, and the
    codes are well formed."""
    make_tabs, ticks, policy, fill, opts, _ = CASES[case]
    tabs = make_tabs()
    B = tabs.shape[0]
    scene = make(backend, B, factored_obs=True, **opts)
    if "threads" in opts:
        assert scene.threads == opts["threads"] and not scene.launch_info["dual"]
    if case == "dual_4096":
        assert scene.launch_info["dual"]
    scene.reset(tabs, warmup=True)
    rng = np.random.RandomState(7)
    check = Checker()
    peak = np.zeros(2, int)                  # most vehicles / agents of an intersection in a tick
    for t in range(ticks):
        pre = before_step(scene)
        out = scene.step(actions_for(scene, rng, policy, t, fill))
        n = out.n_agents
        peak = np.maximum(peak, [int(pre["lane_n"].sum(dim=1).max()), int((out.agent_offset[1:] - out.agent_offset[:-1]).max())])
        check(out, pre, n, what="%s tick %d" % (case, t))
    assert scene.stats()["overflow"] == 0
    assert check.prev_coded > 0
    if "agent_cap" in opts:      # the batch outgrows the next smaller class
        small = {80: (96, 64), 96: (96, 64), 128: (128, 96), 320: (192, 128), 416: (384, 320)}[opts["agent_cap"]]
        assert peak[0] > small[0] or peak[1] > small[1], (peak, small)


@pytest.mark.parametrize("backend", BACKENDS)
def test_without_obs_everything_else_is_identical(backend):
    """``full_obs=False`` (the 784-byte block is not written): every other output, the neighbour sources, the state and
    the statistics are bit-identical to a twin scene with the default outputs, and the expansion is the twin's ``obs``."""
    B = 4
    tabs = mixed_tables(B, 1400, 9)
    twin = make(backend, B, neighbour_sources=True)
    fact = make(backend, B, neighbour_sources=True, factored_obs=True, full_obs=False)
    assert fact.out.obs is None
    for sc in (twin, fact):
        sc.reset(tabs, warmup=True)
    rng = np.random.RandomState(3)
    for t in range(300):
        a = actions_for(twin, rng, "uniform", t, 0)
        o1, o2 = twin.step(a), fact.step(a.clone())
        n = o1.n_agents
        assert o2.n_agents == n
        for f in ("agent_offset", "env_collisions", "env_lock", "env_removed"):
            assert torch.equal(getattr(o1, f), getattr(o2, f)), (t, f)
        for f in ("reward", "ids", "cpv", "status", "jerk_sum", "nbr_src"):
            x, y = getattr(o1, f)[:n], getattr(o2, f)[:n]
            assert torch.equal(bits(x) if x.dtype == torch.float32 else x, bits(y) if y.dtype == torch.float32 else y), (t, f)
        assert_bits_equal(o2.expand_obs(), o1.obs[:n], "tick %d" % t)
    s1, s2 = twin.get_state(), fact.get_state()
    for k in s1:
        np.testing.assert_array_equal(s1[k], s2[k], err_msg=k)
    assert torch.equal(twin.env_stats().clone(), fact.env_stats().clone())
    assert twin.stats() == fact.stats()


def test_nstep_push_refuses_outputs_without_obs():
    from pve_mcc_for_unsignalized_intersection_b200.nstep import NStepFolder
    scene = make("emul", 2, factored_obs=True, full_obs=False)
    folder = NStepFolder.__new__(NStepFolder)        # push checks its argument before it touches the handle
    folder.scene = scene
    with pytest.raises(ValueError, match="full_obs=False"):
        folder.push(scene.out, 0.8)


@pytest.mark.parametrize("backend", BACKENDS)
def test_teacher_forcing(backend):
    """After ``set_state`` with oracle states the expansion is still ``obs`` and ``prev_row0`` the forced rows."""
    B = 4
    tabs = synthetic_arrivals(B, 1200, 45.0, seed=23, rows=40)
    scene = make(backend, B, factored_obs=True)
    orc = P.make_oracle(B, vm=5, veh_cap=scene.veh_cap)
    scene.reset(tabs, warmup=True)
    orc.reset(tabs, warmup=True)
    rng = np.random.RandomState(8)
    check = Checker()
    forced = 0
    for t in range(200):
        orc.step(P.random_actions(rng, orc.control_mask()))            # the oracle runs its own actions
        force = t % 25 == 0
        if force:
            scene.set_state(P.oracle_state_for_device(orc.get_state()))
            forced += 1
        pre = before_step(scene)
        out = scene.step(actions_for(scene, rng, "uniform", t, 0))
        check(out, pre, out.n_agents, continuity=not force, what="tick %d" % t)
    assert forced == 8 and check.prev_coded > 0


@pytest.mark.parametrize("backend", BACKENDS)
def test_out_cap_too_small(backend):
    """The intersections whose rows do not fit ``out_cap`` get none of their factored rows written, and nothing lands
    past ``out_cap`` (the buffers here are longer than the scene's ``out_cap``)."""
    B, cap, guard = 8, 120, 80
    tabs = synthetic_arrivals(B, 1000, 40.0, seed=21, rows=32)
    scene = make(backend, B, out_cap=cap, factored_obs=True)
    scene.out = StepOutputs(B, cap + guard, scene.device, factored=True, lib=scene.lib)
    scene._out_native = scene.out.native()
    scene.reset(tabs, warmup=True)
    rng = np.random.RandomState(3)
    suppressed = 0
    for t in range(200):
        for f in ("row0_out", "prev_row0", "obs"):
            getattr(scene.out, f).view(torch.int32).fill_(0x7FBADBAD)
        scene.out.obs_src.fill_(0x5A5A)
        pre = before_step(scene)
        out = scene.step(actions_for(scene, rng, "uniform", t, 0))
        off = out.agent_offset.to(torch.int64).cpu()
        fits = off[1:] <= cap
        last = int(off[1:][fits].max()) if bool(fits.any()) else 0        # rows of the intersections that fit
        assert bool((off[:-1][fits] <= cap).all())
        suppressed += int((~fits).sum())
        sub = StepOutputs.__new__(StepOutputs)                            # the written rows: check them like any tick
        sub.__dict__.update(out.__dict__)
        sub.agent_offset = torch.minimum(out.agent_offset, torch.tensor(last, dtype=torch.int32, device=out.agent_offset.device))
        Checker()(sub, pre, last, what="tick %d" % t)
        assert bool((out.obs_src[last:] == 0x5A5A).all())
        for f in ("row0_out", "prev_row0"):
            assert bool((getattr(out, f)[last:].view(torch.int32) == 0x7FBADBAD).all()), (t, f)
        # the expanders skip the intersections that do not fit the cap: rows from `last` on stay as they were
        full = torch.full((cap + guard, 7, 28), 7.0, device=scene.device)
        out.expand_obs(n=cap, out=full)
        assert bool((full[last:] == 7.0).all())
        assert_bits_equal(full[:last], out.obs[:last], "tick %d, expansion under the cap" % t)
    assert suppressed > 50 and scene.stats()["overflow"] > 0


def host_copy(out):
    """A host StepOutputs holding the factored block (and obs) of ``out``."""
    h = StepOutputs(out.B, out.out_cap, "cpu", factored=True, lib=out._lib)
    for f in ("agent_offset", "row0_out", "prev_row0", "obs_src", "obs"):
        getattr(h, f).copy_(getattr(out, f).cpu())
    h._n = out.n_agents
    return h


@pytest.mark.parametrize("backend", BACKENDS)
def test_host_expander_threads_and_corruption(backend):
    """Chunked over intersection ranges from several threads the host expander equals one whole call (and ``obs``);
    a corrupted code array is reported, and nothing outside the rows is written."""
    B = 16
    tabs = mixed_tables(B, 1400, 12)
    scene = make(backend, B, factored_obs=True)
    scene.reset(tabs, warmup=True)
    rng = np.random.RandomState(4)
    for t in range(150):
        scene.step(actions_for(scene, rng, "uniform", t, 0))
    h = host_copy(scene.out)
    n = h.n_agents
    whole = h.expand_obs(threads=1).clone()
    assert_bits_equal(whole, h.obs[:n], "host expander")
    for threads in (2, 4, 16, 40):
        assert_bits_equal(h.expand_obs(threads=threads), whole, "%d threads" % threads)
    # arbitrary ranges straight through the C entry point, from a pool of threads
    lib = h._lib
    off_ptr = h.agent_offset.data_ptr()
    ptrs = (h.row0_out.data_ptr(), h.prev_row0.data_ptr(), h.obs_src.data_ptr())
    dst = torch.full((h.out_cap, 7, 28), float("nan"))
    cuts = sorted(set([0, B] + list(rng.randint(0, B, size=5))))
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(4) as pool:
        res = list(pool.map(lambda r: lib.pve_expand_obs_host(off_ptr, r[0], r[1], h.out_cap, *ptrs, dst.data_ptr()),
                            zip(cuts[:-1], cuts[1:])))
    assert res == [0] * (len(cuts) - 1)
    assert_bits_equal(dst[:n], whole, "C expander over ranges")
    assert lib.pve_expand_obs_host(off_ptr, 3, 2, h.out_cap, *ptrs, dst.data_ptr()) < 0
    # corrupted codes: out of the intersection's range, past the 14-bit index, a negative code other than -1
    off = h.agent_offset.numpy()
    b = int(np.argmax(np.diff(off)))
    A = int(off[b + 1] - off[b])
    bad = h.obs_src.clone()
    r = int(off[b])
    bad[r, 1] = A
    bad[r, 2] = PREV | A
    bad[r + 1, 3] = 0x3FFF
    bad[r + 1, 4] = -2
    bad[r + 1, 5] = -32768
    corrupt = host_copy(scene.out)
    corrupt.obs_src.copy_(bad)
    guard = torch.full((n + 8, 7, 28), 3.0)
    with pytest.raises(ValueError, match="5 invalid"):
        corrupt.expand_obs(out=guard)
    assert bool((guard[n:] == 3.0).all())
    assert bool(torch.isnan(guard[r, 1]).all()) and bool(torch.isnan(guard[r + 1, 5]).all())
    # offsets that are not a valid scan: negative / decreasing ones count, the rest is skipped
    corrupt.obs_src.copy_(h.obs_src)
    corrupt.agent_offset[1] = -5
    assert lib.pve_expand_obs_host(corrupt.agent_offset.data_ptr(), 0, 2, h.out_cap, corrupt.row0_out.data_ptr(),
                                   corrupt.prev_row0.data_ptr(), corrupt.obs_src.data_ptr(), guard.data_ptr()) == 2


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("lane_num", [4, 8])
def test_lane4_and_lane8_refuse_the_factored_fields(backend, lane_num):
    B = 2
    with pytest.raises(ValueError, match="12-lane"):
        make(backend, B, lane_num=lane_num, factored_obs=True)
    scene = make(backend, B, lane_num=lane_num)
    tabs = synthetic_arrivals(B, 1000, 20.0, seed=1, rows=16)[:, :, :lane_num].copy()
    scene.reset(tabs, warmup=True)
    a = torch.zeros(B, scene.veh_cap, dtype=torch.float32, device=scene.device)
    scene.step(a)
    scene.out = StepOutputs(B, scene.out_cap, scene.device, factored=True, lib=scene.lib)
    scene._out_native = scene.out.native()
    with pytest.raises(N.NativeError, match="12-lane intersection only"):
        scene.step(a)


@pytest.mark.parametrize("backend", BACKENDS)
def test_partial_factored_fields_are_refused(backend):
    scene = make(backend, 2, factored_obs=True)
    scene.reset(synthetic_arrivals(2, 1000, 20.0, seed=1, rows=16), warmup=True)
    scene._out_native.prev_row0 = None
    with pytest.raises(N.NativeError, match="2 of 3"):
        scene.step(torch.zeros(2, scene.veh_cap, dtype=torch.float32, device=scene.device))


# ---- device only ----------------------------------------------------------------------------------------------------
@GPU
def test_device_expander_equals_host_expander():
    B = 512
    tabs = synthetic_arrivals(B, 1000, 40.0, seed=31)
    scene = make("cuda", B, factored_obs=True)
    scene.reset(tabs, warmup=True)
    rng = np.random.RandomState(2)
    for t in range(120):
        out = scene.step(actions_for(scene, rng, "uniform", t, 0))
        if t % 10 == 9:
            n = out.n_agents
            dev = out.expand_obs()
            assert dev.is_cuda
            assert_bits_equal(dev, out.obs[:n], "device expander, tick %d" % t)
            h = host_copy(out)
            assert_bits_equal(h.expand_obs(threads=4), dev.cpu(), "host expander, tick %d" % t)


@GPU
def test_pipelined_host_path_with_factored_copies():
    """``step_host_async`` over its three buffer sets: copy_factored (bit 2) on every tick, with the full observation
    (bit 1) too on some; every delivered tick expands to a twin scene's ``obs``.  Host buffers are overwritten with
    garbage once read, so a short copy shows."""
    B, ticks = 8, 240
    tabs = synthetic_arrivals(B, 1200, 40.0, seed=15, rows=40)
    scene = make("cuda", B, factored_obs=True, full_obs=False)
    twin = make("cuda", B)
    for sc in (scene, twin):
        sc.reset(tabs, warmup=True)
    pairs = scene.make_async_buffers(factored=True, full_obs=True)
    lean = scene.make_async_buffers(factored=True)           # device buffers without obs: the step skips the block
    assert lean[0][0].obs is None and lean[0][1].obs is None
    acts = [torch.zeros(B, scene.veh_cap, dtype=torch.float32).pin_memory() for _ in range(3)]
    rng = np.random.RandomState(5)
    want, sent = [], []
    delivered = 0

    def take():
        nonlocal delivered
        n, h = scene.host_wait()
        w_obs, with_obs = want.pop(0), sent.pop(0)
        assert n == len(w_obs)
        assert_bits_equal(h.expand_obs(threads=2), w_obs, "delivered tick %d" % delivered)
        if with_obs:
            assert_bits_equal(h.obs[:n], w_obs, "bit 1, tick %d" % delivered)
        for f in ("row0_out", "prev_row0"):
            getattr(h, f).view(torch.int32).fill_(0x7FBADBAD)
        h.obs_src.fill_(0x5A5A)
        delivered += 1

    for t in range(ticks):
        ctrl = twin.control_mask().cpu().numpy()
        a = P.random_actions(rng, ctrl)
        buf = acts[t % 3]
        buf.copy_(torch.from_numpy(a))
        o = twin.step(P.to_device_actions(twin, a))
        want.append(o.obs[:o.n_agents].cpu().clone())
        with_obs = t % 4 == 1
        use = pairs if (t // 3) % 2 == 0 or with_obs else lean
        scene.step_host_async(buf, use[t % 3], copy_obs=with_obs, copy_factored=True)
        sent.append(with_obs)
        if t >= 2:
            take()
    while want:
        take()
    assert delivered == ticks
    with pytest.raises(N.NativeError):          # bit 2 without the factored buffers
        scene.step_host_async(acts[0], scene.make_async_buffers()[0], copy_factored=True)
