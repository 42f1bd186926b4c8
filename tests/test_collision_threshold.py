"""Collision decisions at the threshold, and the step on a non-default geometry, against the float64 oracle.

Phase G3 of the 12-lane step (csrc/scene_step.cuh) decides a collision from world positions computed in float32
(``pve_world_xy_f32``, ``__sincosf`` on the device) and redoes the pair in float64 (``pve_collide_exact``) only when the
float32 distance lies within ``PVE_XY_MARGIN`` (2 cm) of ``collision_thr``.  Every decision must still be the float64
one.  The tests here put one pair of agents per intersection at a float64 world distance of ``thr + delta`` after the
step, for deltas on both sides of the margin and down to 1e-9 m, on every branch of ``get_p`` and at its branch edges,
and compare one tick of every 12-lane kernel variant with the oracle bit for bit.

|delta| < 1e-12 is left out on purpose: the exact path uses CUDA's double ``sincos``, which is not bit-identical to the
libm ``sin`` / ``cos`` of the oracle, so a pair that close to the threshold may be decided either way.

The last part runs free rollouts on a geometry where every ``SceneConfig`` parameter that reaches the step differs from
its default, on 12, 8 and 4 lanes, against oracles that derive their own constants from the same parameters.
"""
import functools
import math
import os
import sys

import numpy as np
import pytest

import parity as P
import test_kernel4_logic_emul as E4
from golden_io import snapshot_to_state
from oracle.oracle import OracleScene, scene_params
from oracle.scene4_oracle import Scene4Oracle
from oracle.scene8_oracle import Scene8Oracle
from pve_mcc_for_unsignalized_intersection_b200 import SceneConfig
from pve_mcc_for_unsignalized_intersection_b200 import _native as N
from pve_mcc_for_unsignalized_intersection_b200.arrivals import synthetic_arrivals
from pve_mcc_for_unsignalized_intersection_b200.config import LANE2LANE
from pve_mcc_for_unsignalized_intersection_b200.scene import BatchedScene

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import make_golden as MG  # noqa: E402  (crafted-state helpers of crafted.npz)

GPU = pytest.mark.gpu
BACKENDS = ["emul", pytest.param("cuda", marks=GPU)]

#: SceneConfig / scene_params arguments besides vm and collision_thr; "wide" changes every one that reaches the step
GEOMETRIES = {"default": {}, "wide": dict(lane_cw=3.5, dis_ctl=180, vM=15, am=-4, aM=2.5, v0=9)}
VM = 5
DELTAS = (-0.5, -0.0201, -0.0199, -1e-3, -1e-6, -1e-9, 1e-9, 1e-6, 1e-3, 0.0199, 0.0201, 0.5)
V_PAIR = 12.0       # both vehicles of a pair: equal speeds keep the rear-end rule (TIS:1509-1516) quiet
P_LOW = -1.0        # lowest post-step position of a pair vehicle: it was at p > 0 before the step, as an agent is
CAP = 128           # vehicle slots of the oracle's state; widened for the larger classes
FAR = np.full((64, 12), 1e6)        # an arrival table with nothing due
FILLER_EVERY = 4    # every 4th intersection also holds 108 uncontrolled vehicles past the exit: the dual mode's big class


def make_scene(backend, B, cfg, veh_cap=128, agent_cap=96, threads=0, neighbour_sources=False):
    if backend == "cuda":
        return BatchedScene(B, cfg, veh_cap=veh_cap, agent_cap=agent_cap, device="cuda:0", threads=threads,
                            neighbour_sources=neighbour_sources)
    from emul.build_emul import build_emul
    return BatchedScene(B, cfg, veh_cap=veh_cap, agent_cap=agent_cap, device="cpu", _library=build_emul(),
                        neighbour_sources=neighbour_sources)


def configs(geometry, thr):
    """(SceneConfig, oracle parameters) of one geometry and threshold."""
    g = GEOMETRIES[geometry]
    return SceneConfig(vm=VM, collision_thr=thr, **g), scene_params(vm=VM, collision_thr=thr, **g)


# ---- 1. the float64 reference of the geometry -----------------------------------------------------------------------
def world_xy12(prm, p, lane):
    """TIS:1250-1290 ``get_p`` for lane_num = 12 in float64, as oracle/scene_oracle.c ``world_xy`` writes it: pi as
    3.141593 (TIS:1259, 1277) and the rotation of ``scene_params`` (TIS:1251, 1287-1288)."""
    cw, m = prm.lane_cw, lane % 3
    if m == 1:
        tx, ty = p - 6 * cw, 3 * cw                                                       # TIS:1270
    else:
        L = prm.lane_len[m]
        if p > L:
            tx, ty = p - L + 6 * cw, (cw if m == 0 else 5 * cw)                           # TIS:1256, 1274
        elif p > 0:
            r_a = (L - p) / L * 3.141593 / 2                                              # TIS:1259, 1277
            c, s = math.cos(r_a), math.sin(r_a)
            if m == 0:
                p0x, p0y, prx, pry = 6 * cw, cw, 6 * cw, -6 * cw
                tx = prx + (p0x - prx) * c - (p0y - pry) * s                              # TIS:1262
                ty = pry + (p0y - pry) * c + (p0x - prx) * s                              # TIS:1263
            else:
                p0x, p0y, prx, pry = 6 * cw, 5 * cw, 6 * cw, 6 * cw
                tx = prx + (p0x - prx) * c + (p0y - pry) * s                              # TIS:1281
                ty = pry + (p0y - pry) * c - (p0x - prx) * s                              # TIS:1282
        elif m == 0:
            tx, ty = -cw, -6 * cw + p                                                     # TIS:1267
        else:
            tx, ty = 5 * cw, 6 * cw - p                                                   # TIS:1286
    c, s = prm.rot_cos[lane // 3], prm.rot_sin[lane // 3]
    return tx * c - ty * s, ty * c + tx * s                                               # TIS:1287-1288


def world_dist(prm, pa, la, pb, lb):
    ax, ay = world_xy12(prm, pa, la)
    bx, by = world_xy12(prm, pb, lb)
    return math.sqrt((bx - ax) * (bx - ax) + (by - ay) * (by - ay))                       # TIS:328


def branch(prm, p, lane):
    """The branch of get_p a vehicle takes: straight lanes have one, turning lanes three."""
    if lane % 3 == 1:
        return "straight"
    return "approach" if p > prm.lane_len[lane % 3] else ("arc" if p > 0 else "exit")


# ---- 2. threshold-straddling pairs ----------------------------------------------------------------------------------
def roots(f, lo, hi, n=240):
    """Every sign change of ``f`` on an ``n``-point grid of [lo, hi], bisected down to adjacent doubles."""
    xs = [float(x) for x in np.linspace(lo, hi, n)]
    fs = [f(x) for x in xs]
    out = []
    for k in range(n - 1):
        if (fs[k] < 0) != (fs[k + 1] < 0):
            a, b, fa = xs[k], xs[k + 1], fs[k]
            while True:
                mid = 0.5 * (a + b)
                if mid in (a, b):
                    break
                fm = f(mid)
                if (fm < 0) == (fa < 0):
                    a, fa = mid, fm
                else:
                    b = mid
            out.append(a if abs(fa) <= abs(f(b)) else b)
    return out


def anchors(prm, lane):
    """Post-step positions of the fixed vehicle of a pair: every branch of get_p, near and far from its edges."""
    L = prm.lane_len[lane % 3]
    if lane % 3 == 1:
        return [-0.6, 0.25 * L, 0.5 * L, 0.8 * L, L + 6.0]
    return [L + 8.0, L + 0.7, 0.8 * L, 0.45 * L, 0.12 * L, -0.6]


def edge_anchors(prm, lane):
    """Post-step positions at the branch edges of get_p, where float32 and float64 can take different branches
    (``(float)p`` rounds onto ``(float)L``; 4e-6 is one or two float32 ulps of L)."""
    L = prm.lane_len[lane % 3]
    u32 = float(np.spacing(np.float32(L)))
    out = [(("L%+g" % d, d), L + d) for d in (1e-12, -1e-12, 4e-6, -4e-6)]
    out += [(("L%+dulp32" % s, s * u32), L + s * u32) for s in (1, -1)]
    return out + [(("0%+g" % d, d), d) for d in (1e-12, -1e-12)]


def candidates(prm, thr):
    """(partner lane, partner p', anchor lane, anchor p', delta, relation, edge label) with the float64 world distance
    of the post-step positions p' equal to thr + delta; the partner's p' is bisected with world_xy12."""
    out = []

    def solve(la, lb, pb, rel, edge):
        hi = prm.lane_len[la % 3] + thr + 30.0
        for d in DELTAS:
            for pa in roots(lambda p: world_dist(prm, p, la, pb, lb) - (thr + d), P_LOW, hi)[:3]:
                out.append((la, pa, lb, pb, d, rel, edge))

    for lb in range(12):
        for pb in anchors(prm, lb):
            solve(lb, lb, pb, "same", None)                                     # followers on the same lane
            if lb % 3 != 2:
                for la in LANE2LANE[lb]:                                        # the conflicting lanes (TIS:153-166)
                    solve(la, lb, pb, "cross", None)
        if lb % 3 != 1:
            for edge, pb in edge_anchors(prm, lb):
                solve(lb, lb, pb, "same", edge)
                if lb % 3 == 0:       # one conflicting lane per approach, a different entry of lane2lane on each
                    solve(LANE2LANE[lb][lb // 3], lb, pb, "cross", edge)
    return out


def build_state(prm, cases, pre):
    """The crafted states: pair vehicles at the pre-step positions ``pre[e] = (p_a, p_b)``, agents at V_PAIR, plus the
    filler of every FILLER_EVERY-th intersection.  Returns the state and the slots of the two vehicles."""
    rng = np.random.RandomState(20261022)
    B = len(cases)
    st, slots = None, np.zeros((B, 2), np.int64)
    for e, (la, _, lb, _, _, _, _) in enumerate(cases):
        s = MG.blank_state()
        vehs = [(la, pre[e][0], 0), (lb, pre[e][1], 1)]
        if e % FILLER_EVERY == FILLER_EVERY - 1:
            vehs += [(lane, -124.0 + 12.0 * k, -1) for lane in range(12) for k in range(9)]
        vehs.sort(key=lambda x: (x[0], x[1]))             # a lane lists its vehicles front (lowest p) first
        for k, (lane, p, who) in enumerate(vehs):
            if who < 0:
                MG.add_veh(s, lane, p, v=prm.v0, control=False)
            else:
                MG.add_veh(s, lane, p, v=V_PAIR)
                slots[e, who] = k
        st = snapshot_to_state(MG.finalize(s, rng), B, CAP, env=e, state=st)
    return st, slots


def oracle_tick(prm, st):
    orc = OracleScene(len(st["tick"]), CAP, prm, n_threads=4)
    orc.reset(FAR, warmup=False)
    orc.set_state(st)
    o = orc.step(np.zeros((len(st["tick"]), CAP), np.float32))
    return o, orc.get_state()


def place(prm, cases):
    """Pre-step positions that the oracle's step moves exactly onto the target post-step positions.  The positions are
    read from an oracle with collision_thr = 0, which moves vehicles as the real one does but removes none of them."""
    B = len(cases)
    cal = scene_params(vm=VM, collision_thr=0, **{k: getattr(prm, k) for k in ("dis_ctl", "vM", "am", "aM", "v0", "lane_cw")})
    target = np.array([(c[1], c[3]) for c in cases])
    pre = target + V_PAIR * prm.dt                            # action 0: the agent keeps its speed on most lanes
    for _ in range(4):
        st, slots = build_state(prm, cases, pre)
        _, post = oracle_tick(cal, st)
        got = np.take_along_axis(post["p"], slots, axis=1)
        if np.array_equal(got, target):
            break
        pre = pre + (target - got)
    assert (pre > 0).all()
    return st, slots, got


def relation(c):
    la, _, lb, _, _, rel, _ = c
    return ("same", la % 3) if rel == "same" else ("cross", la // 3, lb // 3)


@functools.lru_cache(maxsize=None)
def threshold_batch(geometry, thr):
    """The kept pairs of one geometry and threshold: (state, kept cases, oracle outputs, oracle post-tick state)."""
    _, prm = configs(geometry, thr)
    cases = candidates(prm, thr)
    st, slots, got = place(prm, cases)
    o, _ = oracle_tick(prm, st)
    off = o["agent_offset"]
    keep = np.zeros(len(cases), bool)
    for e, c in enumerate(cases):
        pa, pb = got[e]
        d = world_dist(prm, pa, c[0], pb, c[2])
        assert abs(d - (thr + c[4])) <= max(abs(c[4]) / 10, 1e-12), (c, d)
        if c[6] is not None:                                  # the anchor sits at its branch edge, on the intended side
            assert abs(pb - c[3]) <= abs(c[6][1]) / 10, (c, pb)
        # the two agent rows of the intersection (the filler is never an agent) and their nearest neighbours
        ids = [tuple(r) for r in o["ids"][off[e]:off[e + 1]]]
        nn0 = [tuple(r) for r in o["nn"][off[e]:off[e + 1], 0]]
        me = [(c[0], int(slots[e, 0] - st["lane_n"][e, :c[0]].sum())), (c[2], int(slots[e, 1] - st["lane_n"][e, :c[2]].sum()))]
        assert sorted(ids) == sorted(me), (c, ids)
        tested = any(nn0[r] == me[1 - me.index(ids[r])] for r in range(2))       # G3 tests this pair
        hit = bool(o["collisions"][e] > 0)
        if tested:                                            # the oracle decides exactly as this reference does
            assert hit == (d < thr), (c, d, hit)
        else:
            assert not hit, c
        keep[e] = tested
    kept = [c for c, k in zip(cases, keep) if k]
    st = {k: np.ascontiguousarray(v[keep]) for k, v in st.items()}
    o, post = oracle_tick(prm, st)
    check_coverage(prm, kept, o)
    return st, kept, o, post


def coverage(prm, kept, o):
    """Kept pairs per delta, lane relation, branch of each vehicle of a tested pair (the ego of the collision test
    and its neighbour) and branch edge, with the collision outcomes."""
    hit = o["collisions"] > 0
    off = o["agent_offset"]
    cov = {"delta": {}, "outcome": {}, "relation": {}, "branch": {}, "edge": {}}
    for e, c in enumerate(kept):
        la, pa, lb, pb, d, rel, edge = c
        cov["delta"][d] = cov["delta"].get(d, 0) + 1
        cov["outcome"].setdefault(abs(d), set()).add(bool(hit[e]))
        cov["relation"][relation(c)] = cov["relation"].get(relation(c), 0) + 1
        ids = [tuple(r) for r in o["ids"][off[e]:off[e + 1]]]
        nn0 = [tuple(r) for r in o["nn"][off[e]:off[e + 1], 0]]
        # a lane lists its vehicles front (lowest p) first: that orders the two ids of a same-lane pair
        veh = sorted([(la, pa), (lb, pb)])
        for r in range(2):
            other = ids[1 - r]
            if nn0[r] == other:
                for role, (lane, p) in (("ego", veh[sorted(ids).index(ids[r])]), ("neighbour", veh[sorted(ids).index(other)])):
                    k = (role, branch(prm, p, lane))
                    cov["branch"][k] = cov["branch"].get(k, 0) + 1
        if edge is not None:
            cov["edge"].setdefault(edge[0], set()).add(bool(hit[e]))
    return cov


def check_coverage(prm, kept, o):
    """What every threshold batch must hold, so that it cannot shrink silently."""
    cov = coverage(prm, kept, o)
    for d in DELTAS:
        assert cov["delta"].get(d, 0) >= 20, ("few pairs at delta", d, cov["delta"])
    for ad, seen in cov["outcome"].items():                   # collision and no collision at every |delta|
        assert seen == {True, False}, ("one outcome only at |delta|", ad)
    for m in range(3):                                        # followers on the left arc, straight and right arc lanes
        assert cov["relation"].get(("same", m), 0) >= 12 * len(DELTAS) // 2, ("same-lane pairs of movement", m)
    combos = {r[1:] for r in cov["relation"] if r[0] == "cross"}
    assert len(combos) >= 3, ("cross-lane pairs from too few approach combinations", combos)
    for role in ("ego", "neighbour"):
        for b in ("approach", "arc", "exit"):
            assert cov["branch"].get((role, b), 0) >= 12, ("branch", role, b, cov["branch"])
    labels = {lab for lane in (0, 2) for (lab, _), _ in edge_anchors(prm, lane)}
    for lab in labels:
        assert cov["edge"].get(lab) == {True, False}, ("branch edge", lab, cov["edge"].get(lab))


# ---- 3. one tick of every 12-lane kernel variant against the oracle -------------------------------------------------
def widen(st, cap):
    """An oracle state of CAP slots as the state of a scene with ``cap`` slots."""
    out = {}
    for k, v in st.items():
        if v.ndim >= 2 and v.shape[1] == CAP and k not in ("lane_n", "veh_rec", "head_lane", "head_j"):
            w = np.zeros((v.shape[0], cap) + v.shape[2:], v.dtype)
            w[:, :CAP] = v
            v = w
        out[k] = v
    return out


# variant: scene options (default class 128/96; threads=0 is the class's default launch, dual mode for 128/96)
VARIANTS = {"threads_%d" % nt: dict(threads=nt) for nt in (64, 96, 128, 256, 512)}
VARIANTS.update({"dual": dict(), "class_384_320": dict(veh_cap=384, agent_cap=320),
                 "class_576_416": dict(veh_cap=576, agent_cap=416), "neighbour_sources": dict(neighbour_sources=True)})
THRESHOLD_RUNS = [pytest.param("emul", "default", 2.0, None, id="emul-default-thr2"),
                  pytest.param("emul", "wide", 2.3, None, id="emul-wide-thr2.3")]
THRESHOLD_RUNS += [pytest.param("cuda", g, thr, v, marks=GPU, id="cuda-%s-thr%g-%s" % (g, thr, v))
                   for g, thrs in (("default", (2.0, 2.3, 15.0)), ("wide", (2.3,))) for thr in thrs for v in VARIANTS]


@pytest.mark.parametrize("backend,geometry,thr,variant", THRESHOLD_RUNS)
def test_collision_decisions_at_the_threshold(backend, geometry, thr, variant):
    """One tick from the crafted pairs: outputs (cpv, status, collisions, removals, the -10 rewards) and the float64
    state bit for bit against the oracle."""
    st, kept, o, post = threshold_batch(geometry, thr)
    cfg, _ = configs(geometry, thr)
    B = len(kept)
    opts = VARIANTS[variant] if variant else {}
    scene = make_scene(backend, B, cfg, **opts)
    if backend == "cuda":
        info = scene.launch_info
        if "threads" in opts:                                 # an explicit CTA size selects the single-kernel launch
            assert info["dual"] is False and scene.threads == opts["threads"]
        elif "veh_cap" in opts:
            assert (scene.veh_cap, scene.agent_cap, scene.threads) == (opts["veh_cap"], opts["agent_cap"], 512)
            assert info["dual"] is False
        else:
            assert info["dual"] is True
            nv, nc = st["lane_n"].sum(axis=1), ((st["flags"] & 1) != 0).sum(axis=1)
            big = (nv > info["small_veh_cap"]) | (nc > info["small_agent_cap"])
            assert big.any() and not big.all(), "both kernels of the dual launch must have intersections"
    scene.reset(FAR, warmup=False)
    scene.set_state(P.oracle_state_for_device(widen(st, scene.veh_cap)))
    out = P.outputs_to_numpy(scene.step(P.to_device_actions(scene, np.zeros((B, scene.veh_cap), np.float32))))
    what = "%s %s thr=%g %s" % (backend, geometry, thr, variant)
    P.compare_outputs(out, o, what)
    P.compare_states(scene.get_state(), widen(post, scene.veh_cap), what)
    hit = o["collisions"] > 0
    assert hit.any() and not hit.all()
    # an agent that carries a collision at its turn is removed with -10 (TIS:341-348); a partner processed before the
    # test keeps its count for the next tick (Q4)
    assert (o["reward"][o["cpv"] > 0] == -10).all() and (o["n_removed"][hit] >= 1).all() and (o["n_removed"][~hit] == 0).all()


@pytest.mark.parametrize("geometry,thr", [("default", 2.0), ("default", 2.3), ("default", 15.0), ("wide", 2.3)])
def test_threshold_batches_pin_the_reference_to_the_oracle(geometry, thr):
    """Every batch the device tests use, built without a device: the oracle decides every tested pair as world_xy12
    does, and the batch holds its coverage (both asserted while it is built)."""
    _, prm = configs(geometry, thr)
    st, kept, o, _ = threshold_batch(geometry, thr)
    assert len(kept) >= 3000 and len(st["tick"]) == len(kept)
    assert sum(coverage(prm, kept, o)["delta"].values()) == len(kept)


# ---- 4. a non-default geometry, free running ------------------------------------------------------------------------
@pytest.mark.parametrize("backend,threads", [("emul", 0), pytest.param("cuda", 0, marks=GPU),
                                             pytest.param("cuda", 64, marks=GPU)])
def test_free_running_wide_geometry_matches_oracle(backend, threads):
    """12 lanes: random actions for 300 ticks, every tick's outputs and every 20th state against the oracle built from
    the same parameters."""
    cfg, prm = configs("wide", 2.3)
    B = 4 if backend == "emul" else 12
    tabs = synthetic_arrivals(B, 1300, 45.0, seed=31, rows=48)
    scene = make_scene(backend, B, cfg, threads=threads)
    orc = OracleScene(B, scene.veh_cap, prm, n_threads=4)
    scene.reset(tabs, warmup=True)
    orc.reset(tabs, warmup=True)
    rng = np.random.RandomState(32)
    tot = np.zeros(3, np.int64)
    for t in range(300):
        st = orc.get_state()
        act = P.random_actions(rng, (st["flags"] & 1) != 0)
        o_ref = orc.step(act)
        o_dev = P.outputs_to_numpy(scene.step(P.to_device_actions(scene, act)))
        P.compare_outputs(o_dev, o_ref, "wide geometry tick %d" % t)
        if t % 20 == 0 or t == 299:
            P.compare_states(scene.get_state(), orc.get_state(), "wide geometry tick %d" % t)
        tot += [o_ref["collisions"].sum(), o_ref["lock"].sum(), ((o_ref["status"] & N.ST_FINISHED) != 0).sum()]
    assert (tot > 0).all(), ("collisions, lock events, vehicles through", tot)


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("lanes", [4, 8])
def test_free_running_wide_geometry_lane4_and_lane8(backend, lanes, monkeypatch):
    """4 and 8 lanes: ``free_run4`` of tests/test_kernel4_logic_emul.py, with the scene and the Scene4Oracle /
    Scene8Oracle instances it builds given the same parameters."""
    g = dict(GEOMETRIES["wide"], collision_thr=2.3)
    tot = np.zeros(3, np.int64)          # collisions, lock events, vehicles through, summed over the oracles' ticks

    def wide(base):
        class Wide(base):
            def __init__(self, vm=VM):
                super().__init__(vm=vm, **g)

            def step(self, actions):
                r = super().step(actions)
                tot[:] += [r["collisions"], r["lock"], len(r["jerks"])]
                return r
        return Wide

    monkeypatch.setattr(E4, "Scene4Oracle", wide(Scene4Oracle))
    monkeypatch.setattr(E4, "Scene8Oracle", wide(Scene8Oracle))
    built = []
    monkeypatch.setattr(E4, "make_scene4", lambda backend, B, vm=VM, lanes=4:
                        built.append(make_scene(backend, B, SceneConfig(vm=vm, lane_num=lanes, **g))) or built[-1])
    assert E4.free_run4(backend, 3, 1400 if lanes == 4 else 1000, 260, seed=40 + lanes, lanes=lanes) > 3000
    assert len(built) == 1 and built[0].cfg.lane_cw == g["lane_cw"]        # the run used the patched builders
    assert (tot > 0).all(), ("collisions, lock events, vehicles through", tot)
