"""Factored observation outputs at the default workload: step kernel time with and without the 784-byte observation
block, the pipelined host path with the whole observation against the factored one, and the host expansion.

Workload: BASELINE config 2 as bench.py runs it (4 096 intersections, synthetic Poisson arrivals 1 000 veh/h/lane,
actions U(-3, 3), vm 6, 400 priming ticks, L2 flushed between timed ticks).  Variants run on twin scenes fed the same
actions and alternate tick by tick (kernel times) or block by block (host path) within one call.  Prints one JSON
line.  Needs a CUDA device.

    python tools/factored_obs_bench.py [--steps 200] [--envs 4096] [--blocks 4]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (config 2 constants, arrival tables, clock sampler)

PEAK_GBS = 6545.0                  # the HBM bandwidth the roofline of DESIGN.md section 6 is quoted against
OBS_BYTES = 7 * 28 * 4             # one agent's observation
FACT_BYTES = 2 * 28 * 4 + 8 * 2    # row0_out + prev_row0 + obs_src
RECORD_BYTES = 16


def card_info(index):
    info = {"name": None, "power_limit_w": None, "sm_clock_mhz": None, "sm_max_clock_mhz": None}
    import torch
    info["name"] = torch.cuda.get_device_name(index)
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        info["power_limit_w"] = pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
        info["sm_clock_mhz"] = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
        info["sm_max_clock_mhz"] = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
    except Exception as e:           # no NVML binding: say so rather than guess
        info["nvml_error"] = repr(e)
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200, help="timed ticks per variant")
    ap.add_argument("--envs", type=int, default=bench.ENVS_PER_GPU)
    ap.add_argument("--blocks", type=int, default=4, help="host path: alternating blocks of --steps ticks per variant")
    ap.add_argument("--expand-reps", type=int, default=20)
    args = ap.parse_args()

    import torch
    from pve_mcc_for_unsignalized_intersection_b200 import SceneConfig
    from pve_mcc_for_unsignalized_intersection_b200.scene import BatchedScene

    if not torch.cuda.is_available():
        raise SystemExit("factored_obs_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, K = args.envs, args.steps
    ns = argparse.Namespace(workload="poisson", density=bench.DENSITY)
    horizon = (bench.PRIME_TICKS + 3 * K * (2 + args.blocks) + 100) * 0.1 + 30.0
    tabs = bench.make_tables(ns, B, 1000, horizon)
    cfg = lambda: SceneConfig(vm=bench.VM, zero_uncontrolled_actions=True)
    mk = lambda **kw: BatchedScene(B, cfg(), veh_cap=bench.VEH_CAP, agent_cap=bench.AGENT_CAP, device=dev, **kw)
    gen = torch.Generator(device=dev)
    gen.manual_seed(99)
    pool = [(torch.rand(B, bench.VEH_CAP, device=dev, generator=gen) * 6.0 - 3.0).contiguous() for _ in range(16)]
    flush = torch.empty(384 * 1024 * 1024, dtype=torch.uint8, device=dev)
    card = card_info(0)
    sampler = bench.ClockSampler(0)
    sampler.start()

    # ---- 1. step kernel: default / factored + obs / factored without obs, alternating tick by tick ----------------
    variants = {"default": mk(), "factored_with_obs": mk(factored_obs=True), "factored_no_obs": mk(factored_obs=True, full_obs=False)}
    for sc in variants.values():
        sc.reset(tabs, warmup=True)
    for t in range(bench.PRIME_TICKS):
        for sc in variants.values():
            sc.step(pool[t % len(pool)])
    torch.cuda.synchronize()
    for sc in variants.values():
        sc.set_profiling(True)
    kern = {k: [] for k in variants}
    s0 = {k: sc.stats() for k, sc in variants.items()}
    for t in range(K):
        a = pool[t % len(pool)]
        for name, sc in variants.items():
            flush.fill_(t & 0xFF)
            sc.step(a)
            kern[name].append(sc.kernel_ms()[0])
    for sc in variants.values():
        sc.set_profiling(False)
    s1 = {k: sc.stats() for k, sc in variants.items()}
    rows = {k: s1[k]["agent_steps"] - s0[k]["agent_steps"] for k in variants}
    veh = {k: s1[k]["vehicle_steps"] - s0[k]["vehicle_steps"] for k in variants}
    # bit-exactness of the last tick: device expansion of both factored scenes == the default scene's obs
    n = variants["default"].out.n_agents
    ref = variants["default"].out.obs[:n].contiguous().view(torch.int32)
    exact_step = all(torch.equal(variants[k].out.expand_obs().contiguous().view(torch.int32), ref)
                     for k in ("factored_with_obs", "factored_no_obs"))
    agree = all(rows[k] == rows["default"] and veh[k] == veh["default"] for k in variants)
    per_agent = {"default": bench.BYTES_PER_AGENT, "factored_with_obs": bench.BYTES_PER_AGENT + FACT_BYTES,
                 "factored_no_obs": bench.BYTES_PER_AGENT - OBS_BYTES + FACT_BYTES}
    step = {}
    for name in variants:
        ms = float(np.sum(kern[name]))
        byt = (bench.BYTES_PER_VEH * veh[name] + per_agent[name] * rows[name]) / K
        step[name] = {"kernel_ms_per_tick": ms / K, "kernel_ms_median": float(np.median(kern[name])),
                      "algorithmic_bytes_per_tick": byt, "bytes_formula": "%d*V + %d*A" % (bench.BYTES_PER_VEH, per_agent[name]),
                      "achieved_gbs": byt / (ms / K) / 1e6, "frac_of_peak": byt / (ms / K) / 1e6 / PEAK_GBS,
                      "agents_per_tick": rows[name] / K}
    overflow = sum(sc.stats()["overflow"] for sc in variants.values())
    for sc in variants.values():
        sc.close()
    del variants
    torch.cuda.empty_cache()

    # ---- 2. pipelined host path: whole obs (bit 1) against factored (bit 2), alternating blocks --------------------
    s_obs, s_fact = mk(), mk(factored_obs=True, full_obs=False)
    for sc in (s_obs, s_fact):
        sc.reset(tabs, warmup=True)
    for t in range(bench.PRIME_TICKS):
        for sc in (s_obs, s_fact):
            sc.step(pool[t % len(pool)])
    torch.cuda.synchronize()
    bufs = {"obs": s_obs.make_async_buffers(), "factored": s_fact.make_async_buffers(factored=True)}
    scenes = {"obs": s_obs, "factored": s_fact}
    hact = [p.cpu().pin_memory() for p in pool[:4]]
    expand_buf = torch.empty(B * bench.AGENT_CAP, 7, 28, dtype=torch.float32)
    last = {}

    def run(name, n_ticks, t0, expand_threads=0):
        """n_ticks ticks through the pipelined host path, three in flight; returns (rows, seconds)."""
        sc, pairs = scenes[name], bufs[name]
        got = 0
        torch.cuda.synchronize()
        w0 = time.perf_counter()
        for t in range(n_ticks):
            sc.step_host_async(hact[(t0 + t) % len(hact)], pairs[(t0 + t) % 3], copy_obs=name == "obs",
                               copy_factored=name == "factored")
            if t >= 2:
                k, h = sc.host_wait()
                got += k
                if expand_threads:
                    h.expand_obs(out=expand_buf, threads=expand_threads)
                last[name] = (k, h)
        for _ in range(min(2, n_ticks)):
            k, h = sc.host_wait()
            got += k
            if expand_threads:
                h.expand_obs(out=expand_buf, threads=expand_threads)
            last[name] = (k, h)
        return got, time.perf_counter() - w0

    e2e = {"obs": [0, 0.0], "factored": [0, 0.0]}
    tick = 0
    for name in ("obs", "factored"):       # warm-up: every buffer set once
        run(name, 6, tick)
    tick += 6
    for blk in range(args.blocks):
        for name in (("obs", "factored") if blk % 2 == 0 else ("factored", "obs")):
            r, s = run(name, K, tick)
            e2e[name][0] += r
            e2e[name][1] += s
        tick += K
    # the twins got the same actions: the last delivered tick of each must agree bit for bit
    (n_o, h_o), (n_f, h_f) = last["obs"], last["factored"]
    exact_e2e = n_o == n_f and torch.equal(h_f.expand_obs(n_f).contiguous().view(torch.int32),
                                           h_o.obs[:n_o].contiguous().view(torch.int32))
    # host expansion of one delivered tick, per thread count
    expand = {}
    for threads in (1, 4, 16):
        h_f.expand_obs(out=expand_buf, threads=threads)
        w0 = time.perf_counter()
        for _ in range(args.expand_reps):
            h_f.expand_obs(out=expand_buf, threads=threads)
        s = (time.perf_counter() - w0) / args.expand_reps
        expand[str(threads)] = {"ms_per_tick": 1e3 * s, "obs_gbs": n_f * OBS_BYTES / s / 1e9}
    # expansion overlapped with the ticks in flight: every delivered tick expanded before the next wait
    overlapped = {}
    for threads in (4, 16):
        r, s = run("factored", K, tick, expand_threads=threads)
        tick += K
        overlapped[str(threads)] = {"ms_per_tick": 1e3 * s / K, "agent_steps_per_s": r / s}
    sampler.stop_flag = True
    mean_rows = {k: e2e[k][0] / (K * args.blocks) for k in e2e}
    small = (4 * B + 1) * 4
    d2h = {"obs": mean_rows["obs"] * (RECORD_BYTES + OBS_BYTES) + small,
           "factored": mean_rows["factored"] * (RECORD_BYTES + FACT_BYTES) + small}
    line = {
        "tool": "tools/factored_obs_bench.py",
        "card": card, "clocks": sampler.result(),
        "config": {"envs": B, "density": bench.DENSITY, "vm": bench.VM, "prime_ticks": bench.PRIME_TICKS, "steps": K,
                   "blocks": args.blocks, "class": [bench.VEH_CAP, bench.AGENT_CAP], "peak_gbs": PEAK_GBS,
                   "l2": "flushed between timed ticks (384 MiB fill) in the kernel timing; not flushed on the host path"},
        "step_kernel": step,
        "e2e": {k: {"ms_per_tick": 1e3 * e2e[k][1] / (K * args.blocks), "agent_steps_per_s": e2e[k][0] / e2e[k][1],
                    "d2h_bytes_per_tick": d2h[k], "h2d_bytes_per_tick": B * bench.VEH_CAP * 4} for k in e2e},
        "host_expand": expand,
        "e2e_factored_with_overlapped_expand": overlapped,
        "bit_exact": {"step_last_tick": bool(exact_step), "e2e_last_tick": bool(exact_e2e), "twins_agree": bool(agree)},
        "overflow": overflow,
    }
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
