"""The n-step folder with the factored frame log against the full-frame one, on the training workload.

Workload: `bench.py --workload train` (BASELINE config 2 arrivals, 4 096 intersections, class 128/96, vm 5, the
pretrained actor choosing every tick's actions, seq_max_step 12, 400 priming ticks, L2 flushed between timed ticks).
Two variants run on twin scenes and alternate tick by tick within one call:
  full      BatchedScene(neighbour_sources=True), NStepFolder, bind_outputs(), push (pve_nstep_push_scene);
  factored  BatchedScene(factored_obs=True, full_obs=False), NStepFolder(factored=True), bind_outputs(), push
            (pve_nstep_push_factored).
The twins see the same states, so the actor gives both the same actions.  Per variant: CUDA events around actor + step
+ push and around the push, and the library's events around the fold kernel (pve_nstep_set_profiling); the frame-log
bytes of both folders; a bit-for-bit comparison of their replay memories.  Then the same at --big-envs intersections
(the out_cap bench.py uses there: 96 rows per intersection).  The fold's bytes are algorithmic (from shapes); DRAM bytes
are not measured.  Prints one JSON line.  Needs a CUDA device.

    python tools/nstep_factored_bench.py [--steps 100] [--envs 4096] [--big-envs 32768] [--big-steps 30]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402  (config 2 constants, arrival tables, clock sampler)
from factored_obs_bench import card_info  # noqa: E402

FRAME = 7 * 28 * 4                      # one observation block
ROW = 28 * 4
CODES = 8 * 2


def run(B, K, prime):
    import ctypes as C

    import torch
    from pve_mcc_for_unsignalized_intersection_b200 import SceneConfig
    from pve_mcc_for_unsignalized_intersection_b200.actor import ActorWeights, BatchedActor
    from pve_mcc_for_unsignalized_intersection_b200.nstep import BatchedCritic, CriticWeights, NStepFolder
    from pve_mcc_for_unsignalized_intersection_b200.scene import BatchedScene

    dev = torch.device("cuda", 0)
    ns = argparse.Namespace(workload="train", density=bench.DENSITY)
    tabs = bench.make_tables(ns, B, 1000, (prime + 2 * K + 50) * 0.1 + 30.0)
    mk = lambda **kw: BatchedScene(B, SceneConfig(vm=5, zero_uncontrolled_actions=True), veh_cap=bench.VEH_CAP,
                                   agent_cap=bench.AGENT_CAP, device=dev, **kw)
    scenes = {"full": mk(neighbour_sources=True), "factored": mk(factored_obs=True, full_obs=False)}
    actor = BatchedActor(ActorWeights.from_npz(os.path.join(ROOT, "tests", "golden", "actor_agent1.npz")), device=dev)
    with np.load(os.path.join(ROOT, "tests", "golden", "nstep_nets.npz")) as z:
        t_actor = BatchedActor(ActorWeights({k[len("actor__"):].replace("__", "/"): z[k] for k in z.files
                                             if k.startswith("actor__")}), device=dev)
        t_critic = BatchedCritic(CriticWeights({k[len("critic__"):].replace("__", "/"): z[k] for k in z.files
                                                if k.startswith("critic__")}), device=dev)
    folders, bufs = {}, {}
    for name, sc in scenes.items():
        sc.reset(tabs, warmup=True)
        folders[name] = NStepFolder(sc, t_actor, t_critic, seq_max_step=12, buffer_size=max(500000, sc.out_cap + 1),
                                    factored=name == "factored")
        bufs[name] = torch.empty(B, bench.VEH_CAP, dtype=torch.float32, device=dev)
    flush = torch.empty(384 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def tick(name):
        sc, f = scenes[name], folders[name]
        a = actor.act(sc, out=bufs[name])
        f.bind_outputs()
        out = sc.step(a)
        ev[1].record()
        f.push(out, bench.TRAIN_GAMMA)
        return out

    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    for _ in range(prime):
        for name in scenes:
            tick(name)
    torch.cuda.synchronize()
    for f in folders.values():
        f.lib.pve_nstep_set_profiling(f._h, 1)
    ms = {n: {"tick": [], "push": [], "fold": []} for n in scenes}
    rows = {n: 0 for n in scenes}
    records = {n: 0 for n in scenes}
    sampler = bench.ClockSampler(0)
    sampler.start()
    for t in range(K):
        for name in (("full", "factored") if t % 2 == 0 else ("factored", "full")):
            flush.fill_(t & 0xFF)
            ev[0].record()
            out = tick(name)
            ev[2].record()
            ev[2].synchronize()
            fold = C.c_float()
            f = folders[name]
            if f.lib.pve_nstep_fold_ms(f._h, C.byref(fold)) != 0:
                raise RuntimeError("pve_nstep_fold_ms failed")
            ms[name]["tick"].append(ev[0].elapsed_time(ev[2]))
            ms[name]["push"].append(ev[1].elapsed_time(ev[2]))
            ms[name]["fold"].append(fold.value)
            rows[name] += out.n_agents
            records[name] += f.counters()["last_added"]
    sampler.stop_flag = True
    card = card_info(0)
    # the twins must have folded the same memory, bit for bit (the last 200 000 records and the last bootstrap values)
    c = {n: f.counters() for n, f in folders.items()}
    n_exp = c["full"]["num_experiences"]
    idx = torch.arange(max(0, n_exp - 200_000), n_exp, device=dev) % folders["full"].capacity
    same = c["full"]["num_experiences"] == c["factored"]["num_experiences"] and all(
        torch.equal(folders["full"].arrays()[k].index_select(0, idx).view(torch.uint8),
                    folders["factored"].arrays()[k].index_select(0, idx).view(torch.uint8))
        for k in ("state", "action", "reward", "next_state", "done"))
    n_last = scenes["full"].out.n_agents
    same = same and torch.equal(folders["full"].bootstrap_values()[:n_last], folders["factored"].bootstrap_values()[:n_last])
    overflow = sum(sc.stats()["overflow"] for sc in scenes.values())
    res = {"envs": B, "out_cap": scenes["full"].out_cap, "steps": K, "prime_ticks": prime,
           "agents_per_tick": rows["full"] / K, "records_per_push": records["full"] / K,
           "num_experiences": n_exp, "bit_exact": bool(same), "overflow": overflow,
           "clocks": sampler.result()}
    for name in scenes:
        m = {k: np.asarray(v) for k, v in ms[name].items()}
        rec, agents = records[name] / K, rows[name] / K
        # fold kernel, algorithmic bytes per push: per agent row ids 16 + status 1 + reward 4 + q 4 + plan 4 + table entry
        # (key 8, fill 2 read + written, one fidx and one reward written: 28); per record the two frames in and out
        # (+ action 28, reward 4, done 1 out).  Full frames: 2 x 784 in.  Factored: 2 x (16 codes + 8 offsets + 7 rows
        # of 112) in, an upper bound (a zero row reads nothing); rows shared by neighbouring agents count once per record.
        frame_in = FRAME if name == "full" else CODES + 8 + 7 * ROW
        fold_bytes = agents * (16 + 1 + 4 + 4 + 4 + 28) + rec * (2 * frame_in + 2 * FRAME + 28 + 4 + 1)
        res[name] = {"ms_per_tick": float(m["tick"].mean()), "ms_per_tick_median": float(np.median(m["tick"])),
                     "push_ms": float(m["push"].mean()), "push_ms_median": float(np.median(m["push"])),
                     "fold_kernel_ms": float(m["fold"].mean()), "fold_kernel_ms_median": float(np.median(m["fold"])),
                     "fold_algorithmic_bytes_per_push": fold_bytes,
                     "fold_algorithmic_gbs": fold_bytes / (float(m["fold"].mean()) * 1e-3) / 1e9,
                     "frame_log_bytes": folders[name].log_bytes, "card": card}
    res["log_ratio"] = folders["factored"].log_bytes / folders["full"].log_bytes
    for f in folders.values():
        f.lib.pve_nstep_set_profiling(f._h, 0)
        f.close()
    for sc in scenes.values():
        sc.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100, help="timed ticks per variant")
    ap.add_argument("--envs", type=int, default=bench.ENVS_PER_GPU)
    ap.add_argument("--prime", type=int, default=bench.PRIME_TICKS)
    ap.add_argument("--big-envs", type=int, default=32768, help="0: skip the second size")
    ap.add_argument("--big-steps", type=int, default=30)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("nstep_factored_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    line = {"tool": "tools/nstep_factored_bench.py",
            "config": {"workload": "bench.py --workload train (vm 5, pretrained actor, seq_max_step 12, gamma %.6f)"
                                   % bench.TRAIN_GAMMA, "density": bench.DENSITY,
                       "class": [bench.VEH_CAP, bench.AGENT_CAP],
                       "l2": "flushed between timed ticks (384 MiB fill)",
                       "dram_bytes": "not measured (no profiler on the GPU hosts); fold bytes are algorithmic, from shapes"},
            "runs": [run(args.envs, args.steps, args.prime)]}
    torch.cuda.empty_cache()
    if args.big_envs:
        line["runs"].append(run(args.big_envs, args.big_steps, args.prime))
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
