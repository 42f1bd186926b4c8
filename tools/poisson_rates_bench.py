"""Poisson arrivals at a rate per intersection and lane (BatchedScene.reset_poisson(rates)) and the density sweep on
generated traffic (evaluate.evaluate_poisson).  Writes profiles/r03_poisson_rates_bench.json (or --out) and prints it.

1. Regression check of the one-rate Poisson step: step kernel per tick (pve_set_profiling) at BASELINE config 2
   (4 096 intersections, 1 000 veh/h/lane, vm 6, actions U(-3, 3), class 128/96, dual mode), this build against the
   parent build (--parent-lib, built with tools/ab_build.sh), twin scenes with the same traffic alternating tick by
   tick, L2 flushed before every timed tick.  --runs runs of --steps ticks; mean and median of each run.
2. Step kernel per tick of a 4 096-intersection scene split evenly over the seven densities of batch_test, against
   uniform 1 000 veh/h, this build, alternating tick by tick as in 1.
3. Wall time of evaluate_poisson over the seven densities x --envs-per-density intersections x --ticks ticks, and of
   evaluate_tables on seven intersections (one per density, the mirror's tables) over the same ticks, the shape of
   batch_test.
Needs a CUDA device.

    python tools/poisson_rates_bench.py [--parent-lib .ab/libparent.so] [--steps 300] [--runs 5]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402  (config 2 constants, clock sampler)
from factored_obs_bench import card_info  # noqa: E402

SEED = 2024


class _Absent:
    """Stands in for a symbol an older build lacks, so that the loader can declare its prototype; calling it is an
    error."""

    def __init__(self, name):
        self.name = name

    def __call__(self, *args):
        raise RuntimeError("this build has no %s" % self.name)


def parent_scene(path, make):
    """A scene on the parent build, which lacks pve_reset_poisson_rates (never called on it).  The loader gets a
    stand-in for that symbol; every other prototype, pve_reset_poisson's included, is declared on the real function."""
    from pve_mcc_for_unsignalized_intersection_b200 import _native as N
    orig = N.C.CDLL

    class Lib(orig):
        def __getattr__(self, name):
            if name == "pve_reset_poisson_rates":
                stub = _Absent(name)
                setattr(self, name, stub)
                return stub
            return orig.__getattr__(self, name)
    N.C.CDLL = Lib
    try:
        return make(_library=path)
    finally:
        N.C.CDLL = orig


def alternate(scenes, steps, runs, prime):
    """Step kernel ms per tick of every scene, the scenes stepping in turn (rotating order) with the L2 flushed before
    each timed tick; `runs` runs of `steps` ticks.  Also whether every scene's outputs equal the first one's."""
    import torch
    dev = torch.device("cuda", 0)
    B = next(iter(scenes.values())).B
    gen = torch.Generator(device=dev)
    gen.manual_seed(99)
    pool = [(torch.rand(B, bench.VEH_CAP, device=dev, generator=gen) * 6.0 - 3.0).contiguous() for _ in range(16)]
    flush = torch.empty(384 * 1024 * 1024, dtype=torch.uint8, device=dev)
    names = list(scenes)
    for t in range(prime):
        for sc in scenes.values():
            sc.step(pool[t % len(pool)])
    torch.cuda.synchronize()
    for sc in scenes.values():
        sc.set_profiling(True)
    per_run = {k: [] for k in names}
    same = True
    t = prime
    for _ in range(runs):
        kern = {k: [] for k in names}
        for s in range(steps):
            outs = {}
            for name in names[s % len(names):] + names[:s % len(names)]:
                flush.fill_(t & 0xFF)
                outs[name] = scenes[name].step(pool[t % len(pool)])
                kern[name].append(scenes[name].kernel_ms()[0])
            n = outs[names[0]].n_agents
            same = same and all(o.n_agents == n and torch.equal(o.reward[:n], outs[names[0]].reward[:n])
                                for o in outs.values())
            t += 1
        for name in names:
            k = np.asarray(kern[name])
            per_run[name].append({"mean_ms": float(k.mean()), "median_ms": float(np.median(k))})
    for sc in scenes.values():
        sc.set_profiling(False)
    res = {}
    for name in names:
        means = [r["mean_ms"] for r in per_run[name]]
        meds = [r["median_ms"] for r in per_run[name]]
        res[name] = {"runs": per_run[name], "mean_of_run_means_ms": float(np.mean(means)),
                     "median_of_run_medians_ms": float(np.median(meds)),
                     "run_mean_spread": float((max(means) - min(means)) / np.mean(means))}
    st = {k: sc.stats() for k, sc in scenes.items()}
    res["agent_steps_per_tick"] = {k: s["agent_steps"] / max(s["env_steps"] / B, 1) for k, s in st.items()}
    res["overflow"] = {k: s["overflow"] for k, s in st.items()}
    return res, same


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", default=os.path.join(ROOT, ".ab", "libparent.so"),
                    help="libpve_mcc.so of the parent build for 1 ('' : skip 1)")
    ap.add_argument("--steps", type=int, default=300, help="timed ticks per run and scene")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--envs", type=int, default=bench.ENVS_PER_GPU)
    ap.add_argument("--envs-per-density", type=int, default=64)
    ap.add_argument("--ticks", type=int, default=36000, help="evaluation ticks (batch_test: 36 000)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_poisson_rates_bench.json"))
    args = ap.parse_args()

    import torch
    from pve_mcc_for_unsignalized_intersection_b200 import SceneConfig
    from pve_mcc_for_unsignalized_intersection_b200.actor import ActorWeights
    from pve_mcc_for_unsignalized_intersection_b200.arrivals import poisson_arrivals
    from pve_mcc_for_unsignalized_intersection_b200.evaluate import DENSITIES, evaluate_poisson, evaluate_tables
    from pve_mcc_for_unsignalized_intersection_b200.scene import BatchedScene

    if not torch.cuda.is_available():
        raise SystemExit("poisson_rates_bench.py needs a CUDA device")
    if args.parent_lib and not os.path.exists(args.parent_lib):
        raise SystemExit("%s is missing: build the parent commit's library with `tools/ab_build.sh parent` in a checkout of "
                         "it and copy it here, or pass --parent-lib '' to skip the regression check" % args.parent_lib)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, RATE = args.envs, float(bench.DENSITY)
    mk = lambda **kw: BatchedScene(B, SceneConfig(vm=bench.VM, zero_uncontrolled_actions=True), veh_cap=bench.VEH_CAP,
                                   agent_cap=bench.AGENT_CAP, device=dev, **kw)
    card = card_info(0)
    sampler = bench.ClockSampler(0)
    sampler.start()

    # ---- 1. the one-rate Poisson step against the parent build ------------------------------------------------------
    regression = None
    if args.parent_lib:
        scenes = {"this": mk(), "parent": parent_scene(args.parent_lib, mk)}
        for sc in scenes.values():
            sc.reset_poisson(RATE, SEED, warmup=True)
        assert scenes["this"].launch_info["dual"]
        regression, same = alternate(scenes, args.steps, args.runs, bench.PRIME_TICKS)
        regression["outputs_equal"] = bool(same)
        regression["this_over_parent"] = {
            "mean": regression["this"]["mean_of_run_means_ms"] / regression["parent"]["mean_of_run_means_ms"],
            "median": regression["this"]["median_of_run_medians_ms"] / regression["parent"]["median_of_run_medians_ms"]}
        for sc in scenes.values():
            sc.close()
        del scenes
        torch.cuda.empty_cache()

    # ---- 2. seven densities in one scene against uniform 1 000 veh/h ------------------------------------------------
    dens = np.asarray(DENSITIES, np.float64)
    mixed_rates = dens[np.arange(B) * len(dens) // B][:, None]
    scenes = {"uniform_1000": mk(), "seven_densities": mk()}
    scenes["uniform_1000"].reset_poisson(RATE, SEED, warmup=True)
    scenes["seven_densities"].reset_poisson(mixed_rates, SEED, warmup=True)
    mixed, _ = alternate(scenes, args.steps, args.runs, bench.PRIME_TICKS)
    mixed["seven_over_uniform_median"] = (mixed["seven_densities"]["median_of_run_medians_ms"]
                                          / mixed["uniform_1000"]["median_of_run_medians_ms"])
    mixed["intersections_per_density"] = np.bincount(np.arange(B) * len(dens) // B).tolist()
    for sc in scenes.values():
        sc.close()
    del scenes
    torch.cuda.empty_cache()

    # ---- 3. the density sweep -----------------------------------------------------------------------------------------
    w = ActorWeights.from_npz(os.path.join(ROOT, "tests", "golden", "actor_agent1.npz"))
    evaluate_poisson(w, envs_per_density=2, ticks=200)                       # module load, actor set-up
    torch.cuda.synchronize()
    w0 = time.perf_counter()
    res = evaluate_poisson(w, envs_per_density=args.envs_per_density, ticks=args.ticks, seed=1)
    torch.cuda.synchronize()
    t_poisson = time.perf_counter() - w0
    rows = 64
    while True:
        sec, _ = poisson_arrivals(len(dens), dens[:, None], rows, seed=1)
        if sec[:, -1, :].min() > args.ticks * 0.1 + sec[:, 0, :].min(axis=1).max() + 1.0:
            break
        rows *= 2
    torch.cuda.synchronize()
    w0 = time.perf_counter()
    evaluate_tables(list(sec), w, ticks=args.ticks, veh_cap=192, agent_cap=128)
    torch.cuda.synchronize()
    t_tables = time.perf_counter() - w0
    sweep = {"densities": list(DENSITIES), "envs_per_density": args.envs_per_density, "ticks": args.ticks,
             "evaluate_poisson_s": t_poisson, "evaluate_tables_7_intersections_s": t_tables,
             "reports": {str(r["density"]): r["report"] for r in res}}

    sampler.stop_flag = True
    line = {
        "tool": "tools/poisson_rates_bench.py", "card": card, "clocks": sampler.result(),
        "config": {"envs": B, "rate_veh_per_hour_lane": RATE, "vm": bench.VM, "prime_ticks": bench.PRIME_TICKS,
                   "steps_per_run": args.steps, "runs": args.runs, "class": [bench.VEH_CAP, bench.AGENT_CAP],
                   "parent_lib": args.parent_lib or None,
                   "l2": "flushed (384 MiB fill) before every timed step-kernel tick"},
        "regression_uniform_poisson_step": regression, "seven_densities_step": mixed, "density_sweep": sweep,
    }
    text = json.dumps(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text, flush=True)


if __name__ == "__main__":
    main()
