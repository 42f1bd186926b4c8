"""Device-generated Poisson arrivals (BatchedScene.reset_poisson) against the spawn table they replace.

1. Step kernel (pve_set_profiling) and pve_rollout per tick at BASELINE config 2 (4 096 intersections, 1 000 veh/h/lane,
   vm 6, actions U(-3, 3), class 128/96) on twin scenes with IDENTICAL traffic: the table twin is fed
   to_spawn_ticks(poisson_arrivals(...)).  Step kernel: alternating tick by tick, L2 flushed before every timed tick.
   Rollout: alternating blocks, CUDA events around each block.  The twins must end bit-exact.
2. Reset for a 36 000-tick (3 600 s) horizon at 4 096 and 32 768 intersections: the table path as a user runs it
   (synthetic_arrivals + to_spawn_ticks on the host, upload, pve_reset) against reset_poisson (first call: builds and
   uploads the clock table; later calls: kernels only), with the device bytes each adds (cudaMemGetInfo deltas).
3. Poisson alone at 262 144 intersections: reset and a few ticks; the table it replaces is stated as computed.
Prints one JSON line.  Needs a CUDA device.

    python tools/poisson_arrivals_bench.py [--steps 300] [--rollout-blocks 4] [--big 262144]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (config 2 constants, clock sampler)
from tools.factored_obs_bench import card_info  # noqa: E402

HORIZON_TICKS = 36000          # the reference's batch_test horizon (3 600 s)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=300, help="timed ticks per variant (step kernel)")
    ap.add_argument("--rollout-ticks", type=int, default=100, help="ticks per pve_rollout block")
    ap.add_argument("--rollout-blocks", type=int, default=4)
    ap.add_argument("--envs", type=int, default=bench.ENVS_PER_GPU)
    ap.add_argument("--reset-envs", type=int, nargs="*", default=[4096, 32768])
    ap.add_argument("--big", type=int, default=262144, help="Poisson alone at this many intersections (0: skip)")
    args = ap.parse_args()

    import torch
    from pve_mcc_for_unsignalized_intersection_b200 import SceneConfig
    from pve_mcc_for_unsignalized_intersection_b200.actor import ActorWeights, BatchedActor
    from pve_mcc_for_unsignalized_intersection_b200.arrivals import poisson_arrivals, synthetic_arrivals, to_spawn_ticks
    from pve_mcc_for_unsignalized_intersection_b200.scene import BatchedScene

    if not torch.cuda.is_available():
        raise SystemExit("poisson_arrivals_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, K, RATE, SEED = args.envs, args.steps, float(bench.DENSITY), 2024
    cfg = lambda: SceneConfig(vm=bench.VM, zero_uncontrolled_actions=True)
    mk = lambda n: BatchedScene(n, cfg(), veh_cap=bench.VEH_CAP, agent_cap=bench.AGENT_CAP, device=dev)
    card = card_info(0)
    sampler = bench.ClockSampler(0)
    sampler.start()
    ev = lambda: torch.cuda.Event(enable_timing=True)

    # ---- 1. step kernel and rollout, twins with identical traffic ------------------------------------------------
    total = bench.PRIME_TICKS + K + args.rollout_ticks * args.rollout_blocks + 50
    rows = 64
    while True:
        sec, _ = poisson_arrivals(B, RATE, rows, SEED)
        if sec[:, -1, :].min() > sec[:, 0, :].min(axis=1).max() + total * 0.1 + 1.0:
            break
        rows *= 2
    twins = {"table": mk(B), "poisson": mk(B)}
    twins["table"].reset(spawn_ticks=to_spawn_ticks(sec), warmup=True)
    twins["poisson"].reset_poisson(RATE, SEED, warmup=True)
    del sec
    gen = torch.Generator(device=dev)
    gen.manual_seed(99)
    pool = [(torch.rand(B, bench.VEH_CAP, device=dev, generator=gen) * 6.0 - 3.0).contiguous() for _ in range(16)]
    flush = torch.empty(384 * 1024 * 1024, dtype=torch.uint8, device=dev)
    for t in range(bench.PRIME_TICKS):
        for sc in twins.values():
            sc.step(pool[t % len(pool)])
    torch.cuda.synchronize()
    for sc in twins.values():
        sc.set_profiling(True)
    kern = {k: [] for k in twins}
    for t in range(K):
        order = ("table", "poisson") if t % 2 == 0 else ("poisson", "table")
        for name in order:
            flush.fill_(t & 0xFF)
            twins[name].step(pool[t % len(pool)])
            kern[name].append(twins[name].kernel_ms()[0])
    for sc in twins.values():
        sc.set_profiling(False)
    actor = BatchedActor(ActorWeights.random(0))
    roll = {k: [] for k in twins}
    for blk in range(args.rollout_blocks + 1):          # block 0 warms the actor up
        for name in (("table", "poisson") if blk % 2 == 0 else ("poisson", "table")):
            torch.cuda.synchronize()
            e0, e1 = ev(), ev()
            e0.record()
            actor.rollout(twins[name], args.rollout_ticks)
            e1.record()
            e1.synchronize()
            if blk:
                roll[name].append(e0.elapsed_time(e1) / args.rollout_ticks)
    st = {k: sc.get_state() for k, sc in twins.items()}
    exact = all(np.array_equal(np.asarray(st["table"][k]), np.asarray(st["poisson"][k])) for k in st["table"])
    exact = exact and twins["table"].stats() == twins["poisson"].stats()
    exact = exact and torch.equal(twins["table"].env_stats().clone(), twins["poisson"].env_stats().clone())
    stats = twins["poisson"].stats()
    step = {}
    for name in twins:
        k = np.asarray(kern[name])
        step[name] = {"kernel_ms_per_tick": float(k.mean()), "kernel_ms_median": float(np.median(k)),
                      "kernel_ms_p10_p90": [float(np.percentile(k, 10)), float(np.percentile(k, 90))],
                      "rollout_ms_per_tick": float(np.mean(roll[name])), "rollout_block_ms_per_tick": roll[name]}
    step["poisson_over_table"] = {"kernel_mean": step["poisson"]["kernel_ms_per_tick"] / step["table"]["kernel_ms_per_tick"],
                                  "kernel_median": step["poisson"]["kernel_ms_median"] / step["table"]["kernel_ms_median"],
                                  "rollout": step["poisson"]["rollout_ms_per_tick"] / step["table"]["rollout_ms_per_tick"]}
    for sc in twins.values():
        sc.close()
    del twins, pool, sc, flush
    torch.cuda.empty_cache()

    # ---- 2. reset for a 36 000-tick horizon --------------------------------------------------------------------
    def free_bytes():
        torch.cuda.synchronize()
        torch.cuda.empty_cache()          # blocks torch keeps cached would hide an allocation
        return torch.cuda.mem_get_info(dev)[0]

    resets = {}
    for n in args.reset_envs:
        r = {}
        sc = mk(n)                  # Poisson first, on a fresh handle: nothing freed or cached confounds the bytes
        f0 = free_bytes()
        times = []
        for k in range(4):
            torch.cuda.synchronize()
            w0 = time.perf_counter()
            sc.reset_poisson(RATE, seed=100 + k, warmup=True)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - w0)
        # pending arrival times (96 B per intersection) + the clock table (4 000 001 doubles, one per handle) + the
        # [n][veh_cap] float staging buffer of the warm-up tick's actions, which the first warm reset of a handle
        # allocates on either path
        r["poisson"] = {"device_bytes_measured": int(f0 - free_bytes()),
                        "device_bytes_formula": 96 * n + 8 * 4000001 + 4 * n * bench.VEH_CAP,
                        "first_reset_s": times[0], "later_reset_s": float(np.median(times[1:]))}
        torch.cuda.synchronize()
        w0 = time.perf_counter()
        tabs = synthetic_arrivals(n, RATE, HORIZON_TICKS * 0.1, seed=1)
        w1 = time.perf_counter()
        ticks = to_spawn_ticks(tabs)
        w2 = time.perf_counter()
        f0 = free_bytes()
        sc.reset(spawn_ticks=ticks, warmup=True)
        torch.cuda.synchronize()
        w3 = time.perf_counter()
        r["table"] = {"rows": int(tabs.shape[1]), "host_f64_bytes": int(tabs.nbytes), "device_table_bytes": int(ticks.nbytes),
                      "device_bytes_measured": int(f0 - free_bytes()), "synthetic_arrivals_s": w1 - w0,
                      "to_spawn_ticks_s": w2 - w1, "upload_and_reset_s": w3 - w2, "total_s": w3 - w0}
        del tabs, ticks
        sc.close()
        del sc
        torch.cuda.empty_cache()
        resets[str(n)] = r

    # ---- 3. Poisson alone at a size the table does not reach ----------------------------------------------------
    big = None
    if args.big:
        n = args.big
        sc = mk(n)
        f0 = free_bytes()
        torch.cuda.synchronize()
        w0 = time.perf_counter()
        sc.reset_poisson(RATE, seed=7, warmup=True)
        torch.cuda.synchronize()
        t_reset = time.perf_counter() - w0
        used = f0 - free_bytes()
        a = torch.empty(n, bench.VEH_CAP, device=dev)
        for t in range(60):
            sc.step(a.uniform_(-3.0, 3.0))
        torch.cuda.synchronize()
        sc.set_profiling(True)
        ks = []
        for t in range(40):
            sc.step(a.uniform_(-3.0, 3.0))
            ks.append(sc.kernel_ms()[0])
        s = sc.stats()
        mean = 3600.0 / RATE                    # synthetic_arrivals' sizing rule for the 3 600 s horizon
        rows_k = int(HORIZON_TICKS * 0.1 / (1.0 + mean * np.exp(-1.0 / mean)) * 1.25) + 24
        # measured: pending times + clock table + the [n][veh_cap] float staging buffer of the warm-up tick's actions,
        # which the first warm reset of a handle allocates on either path
        big = {"envs": n, "first_reset_s": t_reset, "device_bytes_measured": int(used),
               "device_bytes_formula": 96 * n + 8 * 4000001 + 4 * n * bench.VEH_CAP,
               "kernel_ms_per_tick": float(np.mean(ks)), "agents_last_tick": int(sc.out.n_agents), "overflow": s["overflow"],
               "table_it_replaces_computed_not_measured": {"rows": rows_k, "device_int32_bytes": n * rows_k * 12 * 4,
                                                           "host_f64_bytes": n * rows_k * 12 * 8}}
        sc.close()
    sampler.stop_flag = True
    line = {
        "tool": "tools/poisson_arrivals_bench.py",
        "card": card, "clocks": sampler.result(),
        "config": {"envs": B, "rate_veh_per_hour_lane": RATE, "vm": bench.VM, "prime_ticks": bench.PRIME_TICKS, "steps": K,
                   "rollout_ticks": args.rollout_ticks, "rollout_blocks": args.rollout_blocks,
                   "class": [bench.VEH_CAP, bench.AGENT_CAP], "horizon_ticks": HORIZON_TICKS,
                   "l2": "flushed (384 MiB fill) before every timed step-kernel tick; not flushed around rollout blocks"},
        "step": step, "twins_bit_exact": bool(exact), "overflow": stats["overflow"],
        "agent_steps_per_tick": stats["agent_steps"] / max(stats["env_steps"] / B, 1),
        "reset_36000_ticks": resets, "poisson_alone": big,
    }
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
