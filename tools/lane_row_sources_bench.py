"""Row sources (pve_outputs.nbr_src) on the 4- and 8-lane step, and the distinct-row n-step push they enable.

Workload: `bench.py --workload lane4` / `lane8` (4 096 intersections, 1 000 veh/h/lane, vm 6, actions U(-3, 3) for the
controlled vehicles; class 64/64 for lane_num 4, 128/96 for lane_num 8), on device-generated Poisson arrivals so that
every scene sees the same traffic.  Per geometry, in one process:
  (i)   step kernel per tick without nbr_src: this build against the parent build (--parent-lib), twin scenes;
  (ii)  step kernel per tick with nbr_src against without, same build;
        (the three scenes alternate tick by tick, L2 flushed before every timed tick; outputs compared every tick)
  (iii) the train tick (pretrained actor + step + n-step push, seq_max_step 12, vm 5): pve_nstep_push (target actor
        on all 7 rows of every observation) against pve_nstep_push_scene (once per distinct row), twin scenes
        alternating tick by tick; CUDA events around actor + step + push and around the push; the target-actor rows
        per tick counted from the outputs; the replay memories compared bit for bit.  The networks run the tcgen05
        kernels (PVE_ACTOR_IMPL / PVE_CRITIC_IMPL = tc5 unless set): what the default choice by row count takes for
        every call at this size except the one-row evaluation of the zero row's action, which it would run on
        mma.sync and so give the two pushes different kernels for that row.
Prints one JSON line.  Needs a CUDA device.

    python tools/lane_row_sources_bench.py [--parent-lib PATH] [--steps 200] [--train-steps 100]
"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402  (config constants, clock sampler)
from factored_obs_bench import card_info  # noqa: E402

GEOMETRIES = {4: (64, 64), 8: (128, 96)}
SEED = 2024


def parent_scene(path, make):
    """A scene on an older build, which lacks pve_row0_prev_dev (never called here): the loader's prototype for it is
    pointed at pve_row0_dev so that every other declaration still applies."""
    from pve_mcc_for_unsignalized_intersection_b200 import _native as N
    orig = N.C.CDLL

    class Lib(orig):
        def __getattr__(self, name):
            if name == "pve_row0_prev_dev":
                return orig.__getattr__(self, "pve_row0_dev")
            return orig.__getattr__(self, name)
    N.C.CDLL = Lib
    try:
        return make(_library=path)
    finally:
        N.C.CDLL = orig


def step_kernels(lanes, B, K, prime, parent_lib):
    import torch
    from pve_mcc_for_unsignalized_intersection_b200 import SceneConfig
    from pve_mcc_for_unsignalized_intersection_b200.scene import BatchedScene
    dev = torch.device("cuda", 0)
    vc, ac = GEOMETRIES[lanes]
    mk = lambda **kw: BatchedScene(B, SceneConfig(vm=bench.VM, lane_num=lanes), veh_cap=vc, agent_cap=ac, device=dev, **kw)
    scenes = {"plain": mk(), "src": mk(neighbour_sources=True)}
    if parent_lib:
        scenes["parent"] = parent_scene(parent_lib, mk)
    for sc in scenes.values():
        sc.reset_poisson(float(bench.DENSITY), SEED, warmup=True)
    gen = torch.Generator(device=dev)
    gen.manual_seed(99)
    pool = [(torch.rand(B, vc, device=dev, generator=gen) * 6.0 - 3.0) for _ in range(16)]
    act = {k: torch.empty(B, vc, device=dev) for k in scenes}
    flush = torch.empty(384 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def tick(name, t):
        sc = scenes[name]
        torch.mul(pool[t % len(pool)], sc.control_mask(), out=act[name])
        return sc.step(act[name])

    for t in range(prime):
        for name in scenes:
            tick(name, t)
    torch.cuda.synchronize()
    for sc in scenes.values():
        sc.set_profiling(True)
    kern = {k: [] for k in scenes}
    same, rows = True, 0
    names = list(scenes)
    for t in range(K):
        order = names[t % len(names):] + names[:t % len(names)]
        outs = {}
        for name in order:
            flush.fill_(t & 0xFF)
            outs[name] = tick(name, prime + t)
            kern[name].append(scenes[name].kernel_ms()[0])
        n = outs["plain"].n_agents
        rows += n
        for name in names:
            o = outs[name]
            same = same and o.n_agents == n and all(torch.equal(getattr(o, f)[:n], getattr(outs["plain"], f)[:n])
                                                    for f in ("obs", "reward", "ids", "status", "cpv", "jerk_sum"))
    for sc in scenes.values():
        sc.set_profiling(False)
    stats = {k: sc.stats() for k, sc in scenes.items()}
    same = same and all(s == stats["plain"] for s in stats.values())
    same = same and all(torch.equal(sc.env_stats().clone(), scenes["plain"].env_stats().clone()) for sc in scenes.values())
    res = {"lane_num": lanes, "class": [vc, ac], "envs": B, "steps": K, "prime_ticks": prime, "agents_per_tick": rows / K,
           "outputs_and_stats_bit_exact": bool(same), "overflow": stats["plain"]["overflow"]}
    for name in names:
        k = np.asarray(kern[name])
        res[name] = {"kernel_ms_per_tick": float(k.mean()), "kernel_ms_median": float(np.median(k)),
                     "kernel_ms_p10_p90": [float(np.percentile(k, 10)), float(np.percentile(k, 90))]}
    res["src_over_plain_median"] = res["src"]["kernel_ms_median"] / res["plain"]["kernel_ms_median"]
    if "parent" in scenes:
        res["plain_over_parent_median"] = res["plain"]["kernel_ms_median"] / res["parent"]["kernel_ms_median"]
    for sc in scenes.values():
        sc.close()
    return res


def train_ticks(lanes, B, K, prime):
    import torch
    from pve_mcc_for_unsignalized_intersection_b200 import SceneConfig
    from pve_mcc_for_unsignalized_intersection_b200.actor import ActorWeights, BatchedActor
    from pve_mcc_for_unsignalized_intersection_b200.nstep import BatchedCritic, CriticWeights, NStepFolder
    from pve_mcc_for_unsignalized_intersection_b200.scene import BatchedScene
    dev = torch.device("cuda", 0)
    vc, ac = GEOMETRIES[lanes]
    mk = lambda **kw: BatchedScene(B, SceneConfig(vm=5, zero_uncontrolled_actions=True, lane_num=lanes), veh_cap=vc,
                                   agent_cap=ac, device=dev, **kw)
    scenes = {"push": mk(), "push_scene": mk(neighbour_sources=True)}
    actor = BatchedActor(ActorWeights.from_npz(os.path.join(ROOT, "tests", "golden", "actor_agent1.npz")), device=dev)
    with np.load(os.path.join(ROOT, "tests", "golden", "nstep_nets.npz")) as z:
        t_actor = BatchedActor(ActorWeights({k[len("actor__"):].replace("__", "/"): z[k] for k in z.files
                                             if k.startswith("actor__")}), device=dev)
        t_critic = BatchedCritic(CriticWeights({k[len("critic__"):].replace("__", "/"): z[k] for k in z.files
                                                if k.startswith("critic__")}), device=dev)
    folders, bufs = {}, {}
    for name, sc in scenes.items():
        sc.reset_poisson(float(bench.DENSITY), SEED, warmup=True)
        folders[name] = NStepFolder(sc, t_actor, t_critic, seq_max_step=12, buffer_size=max(500000, sc.out_cap + 1))
        bufs[name] = torch.empty(B, vc, dtype=torch.float32, device=dev)
    flush = torch.empty(384 * 1024 * 1024, dtype=torch.uint8, device=dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]

    def tick(name):
        sc, f = scenes[name], folders[name]
        a = actor.act(sc, out=bufs[name])
        f.bind_outputs()
        out = sc.step(a)
        ev[1].record()
        f.push(out, bench.TRAIN_GAMMA, distinct_rows=(name == "push_scene"))
        return out

    for _ in range(prime):
        for name in scenes:
            tick(name)
    torch.cuda.synchronize()
    ms = {n: {"tick": [], "push": []} for n in scenes}
    rows, distinct = 0, 0
    sampler = bench.ClockSampler(0)
    sampler.start()
    for t in range(K):
        for name in (("push", "push_scene") if t % 2 == 0 else ("push_scene", "push")):
            flush.fill_(t & 0xFF)
            ev[0].record()
            out = tick(name)
            ev[2].record()
            ev[2].synchronize()
            ms[name]["tick"].append(ev[0].elapsed_time(ev[2]))
            ms[name]["push"].append(ev[1].elapsed_time(ev[2]))
            if name == "push_scene":
                # target-actor rows of push_scene: this tick's row 0 of every agent + every distinct stored row some
                # 0x4000 code names (the zero row's action is computed once, when the actor is created)
                n = out.n_agents
                codes = out.nbr_src[:n, 1:7].int()
                old = (codes >= 0) & ((codes & 0x4000) != 0)
                env = out.ids[:n, 0:1].long().expand(-1, 6)
                keys = env[old] * vc + (codes[old] & 0x3FFF).long()
                rows += n
                distinct += int(torch.unique(keys).numel())
    sampler.stop_flag = True
    c = {n: f.counters() for n, f in folders.items()}
    n_exp = c["push"]["num_experiences"]
    idx = torch.arange(max(0, n_exp - 200_000), n_exp, device=dev) % folders["push"].capacity
    same = c["push"] == c["push_scene"] and all(
        torch.equal(folders["push"].arrays()[k].index_select(0, idx).view(torch.uint8),
                    folders["push_scene"].arrays()[k].index_select(0, idx).view(torch.uint8))
        for k in ("state", "action", "reward", "next_state", "done"))
    n_last = scenes["push"].out.n_agents
    same = same and torch.equal(folders["push"].bootstrap_values()[:n_last], folders["push_scene"].bootstrap_values()[:n_last])
    res = {"lane_num": lanes, "class": [vc, ac], "envs": B, "steps": K, "prime_ticks": prime,
           "agents_per_tick": rows / K, "num_experiences": n_exp, "bit_exact": bool(same),
           "overflow": sum(sc.stats()["overflow"] for sc in scenes.values()), "clocks": sampler.result(),
           "target_actor_rows_per_tick": {"push": 7 * rows / K, "push_scene": (rows + distinct) / K,
                                          "push_scene_prev_rows": distinct / K}}
    for name in scenes:
        m = {k: np.asarray(v) for k, v in ms[name].items()}
        res[name] = {"ms_per_tick": float(m["tick"].mean()), "ms_per_tick_median": float(np.median(m["tick"])),
                     "push_ms": float(m["push"].mean()), "push_ms_median": float(np.median(m["push"]))}
    res["push_scene_over_push_median"] = {"tick": res["push_scene"]["ms_per_tick_median"] / res["push"]["ms_per_tick_median"],
                                          "push": res["push_scene"]["push_ms_median"] / res["push"]["push_ms_median"]}
    for f in folders.values():
        f.close()
    for sc in scenes.values():
        sc.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", default=None, help="libpve_mcc.so of the parent build for (i); omitted: no (i)")
    ap.add_argument("--envs", type=int, default=bench.ENVS_PER_GPU)
    ap.add_argument("--steps", type=int, default=200, help="timed ticks per scene, step kernels")
    ap.add_argument("--train-steps", type=int, default=100, help="timed ticks per variant, train tick")
    ap.add_argument("--prime", type=int, default=bench.PRIME_TICKS)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("lane_row_sources_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    for var in ("PVE_ACTOR_IMPL", "PVE_CRITIC_IMPL"):
        os.environ.setdefault(var, "tc5")
    sampler = bench.ClockSampler(0)
    sampler.start()
    steps = [step_kernels(lanes, args.envs, args.steps, args.prime, args.parent_lib) for lanes in GEOMETRIES]
    sampler.stop_flag = True
    line = {"tool": "tools/lane_row_sources_bench.py", "card": card_info(0), "clocks": sampler.result(),
            "config": {"density": bench.DENSITY, "arrivals": "pve_reset_poisson seed %d" % SEED,
                       "step": "vm %d, actions U(-3, 3) x control mask" % bench.VM,
                       "train": "vm 5, pretrained actor, seq_max_step 12, gamma %.6f, bind_outputs, networks actor %s / "
                                "critic %s" % (bench.TRAIN_GAMMA, os.environ["PVE_ACTOR_IMPL"], os.environ["PVE_CRITIC_IMPL"]),
                       "l2": "flushed between timed ticks (384 MiB fill)", "parent_lib": args.parent_lib},
            "step_kernels": steps,
            "train": [train_ticks(lanes, args.envs, args.train_steps, args.prime) for lanes in GEOMETRIES]}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
