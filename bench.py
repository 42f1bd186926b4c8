#!/usr/bin/env python
"""Benchmark of the batched PVE-MCC environment step (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference]

A "step" is one tick (step() for every vehicle + scene_update() + delete_vehicle()) of every
intersection of the batch.  Workload at N = 1: BASELINE config 2 -- 4,096 intersections,
synthetic Poisson arrivals (1000 veh/h/lane; the train-set table is missing from the reference
checkout, SURVEY.md #22), actions U(-3, 3), vm = 6 (train setting, main.py:230).  With N > 1 every
rank runs its own 4,096 intersections (weak scaling, no step-path communication); NCCL is used
only to all-reduce the end-of-rollout statistics and to take the max of the timings.

Reported: `value` = vehicle-agent env-steps/s with inputs resident in HBM (CUDA events, L2
flushed between timed steps); `e2e` = the same metric through the host-buffer C-ABI call with the FULL 9-tuple
delivered to pinned host memory every step (actions H2D; observations + all per-agent outputs D2H) and `e2e_no_obs`
= the same without the observations (a consumer whose policy runs on the device); `roofline` = algorithmic bytes
(68*V + 1028*A, SURVEY.md 8(d)) / step-kernel time against the measured HBM peak;
`cpu_baseline` = the CPU oracle port on the host cores, timed in the same run.

`--impl reference` times the reference algorithm's CPU port (oracle/scene_oracle.c, all host
threads; the reference itself is pure Python and cannot travel to the GPU box).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "vehicle-agent env-steps/sec"
UNIT = "agent-steps/s"
ENVS_PER_GPU = 4096
DENSITY = 1000
VM = 6
PRIME_TICKS = 400          # untimed: fill the intersections to steady-state occupancy
# Capacity class of the run: 128 vehicle slots / 96 agents per intersection (7 CTAs per SM).  At this
# workload the largest agent count seen in 4096 intersections x 800 ticks is 75 (oracle run, DESIGN.md
# section 6).  The tighter 128/80 class (8 CTAs per SM, PVE_BENCH_AGENT_CAP=80) measures ~2% slower: its
# 64-register budget costs more than the extra resident CTA brings.  Should an intersection ever need
# more agents than the class holds, the kernel defers the arrival and counts it in `overflow`, and the
# benchmark then repeats itself with the 128/96 class instead of reporting a flagged run.
VEH_CAP, AGENT_CAP = 128, int(os.environ.get("PVE_BENCH_AGENT_CAP", "96"))
BYTES_PER_VEH, BYTES_PER_AGENT = 68, 1028        # SURVEY.md 8(d) / BASELINE.md section 4
OBS_BYTES = 7 * 28 * 4                           # one agent's observation


TRAIN_GAMMA = 0.8766832904447475          # main.py:227 at epoch 20: tanh(26 / 12) * 0.9


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="graft", choices=["graft", "reference"])
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU, help="intersections per GPU")
    ap.add_argument("--density", type=int, default=DENSITY)
    ap.add_argument("--threads", type=int, default=0, help="CTA size override (64/128/256)")
    ap.add_argument("--workload", default="poisson", choices=["poisson", "stress", "rollout", "train", "lane4", "lane8"],
                    help="poisson: BASELINE config 2 (default); lane4 / lane8: the same on the 4-lane / 8-lane intersection (lane_num=4 / 8, row N3); stress: config 4; rollout: config 5 = the pretrained "
                         "actor evaluated on the GPU every tick + the environment step; train: rollout + the training "
                         "loop's n-step return folding and replay writer (main.py:243-266) on the GPU every tick")
    ap.add_argument("--veh-cap", type=int, default=VEH_CAP, help="capacity class of the run (vehicle slots per intersection)")
    ap.add_argument("--agent-cap", type=int, default=AGENT_CAP, help="capacity class of the run (agents per intersection)")
    ap.add_argument("--out-rows-per-env", type=int, default=0,
                    help="size the dense output arrays for this many agent rows per intersection instead of agent_cap (very "
                         "large batches: the outputs are dense, so the mean count plus a margin is enough; rows that do not "
                         "fit raise `overflow`, which discards the run)")
    ap.add_argument("--traffic-child", action="store_true", help=argparse.SUPPRESS)      # run under ncu by measure_traffic()
    ap.add_argument("--no-traffic", action="store_true", help="skip the ncu child that measures roofline.traffic")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step handed its caller to DIR/<name>.npy "
                         "(float32 / float64, at most 64 MB in all: larger arrays keep a fixed, seeded sample of their "
                         "rows, listed in DIR/<name>_rows.npy); rank 0 only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "graft":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl graft)")
    return args


def lanes_of(args):
    return {"lane4": 4, "lane8": 8}.get(args.workload, 12)


def workload_name(args):
    if args.workload in ("lane4", "lane8"):
        return ("%d %d-lane intersections (lane_num=%d) per GPU, synthetic Poisson arrivals %d veh/h/lane, actions U(-3,3) for "
                "controlled vehicles and 0 for uncontrolled ones (main.py:401-405), vm=%d%s" % (
                    args.envs, lanes_of(args), lanes_of(args), args.density, VM,
                    ", intention draws numpy default_rng(0) (TIS:390)" if args.workload == "lane8" else ""))
    if args.workload == "stress":
        return "stress: headway 1.0 s on all 12 lanes, all-brake policy, %d intersections per GPU" % args.envs
    if args.workload == "train":
        return ("training rollout: %d intersections per GPU, synthetic Poisson arrivals %d veh/h/lane, pretrained actor "
                "+ environment step + n-step folding (seq_max_step 12, target actor once per distinct observation row, target critic) "
                "+ replay writer (500 000 records) on the GPU every tick, vm=5" % (args.envs, args.density))
    if args.workload == "rollout":
        return ("full rollout: %d intersections per GPU, synthetic Poisson arrivals %d veh/h/lane, actions from the "
                "reference's pretrained actor evaluated on the GPU every tick (tests/golden/actor_agent1.npz), vm=5"
                % (args.envs, args.density))
    return ("%d intersections per GPU, synthetic Poisson arrivals %d veh/h/lane, actions U(-3,3) for controlled vehicles "
            "and 0 for uncontrolled ones (main.py:401-405), vm=%d" % (args.envs, args.density, VM))


def make_tables(args, n_envs, seed, horizon_s):
    from pve_mcc_for_unsignalized_intersection_b200.arrivals import stress_arrivals, synthetic_arrivals
    if args.workload == "stress":
        return stress_arrivals(n_envs, horizon_s)
    tabs = synthetic_arrivals(n_envs, args.density, horizon_s, seed=seed)
    return tabs[:, :, :lanes_of(args)].copy() if lanes_of(args) != 12 else tabs


# ---------------------------------------------------------------------------------------------
# CPU legs (oracle port): cpu_baseline inside the default run, and the whole `--impl reference` arm
# ---------------------------------------------------------------------------------------------
def cpu_port_run(args, n_envs, prime, timed_steps, warmup_steps, n_threads, seed=1234):
    """Times the oracle port: `timed_steps` ticks of `n_envs` intersections after priming."""
    if args.workload in ("lane4", "lane8"):
        return cpu_port_run_lane4(args, n_envs, prime, timed_steps, warmup_steps, seed)
    from oracle.oracle import OracleScene, scene_params
    horizon = (prime + warmup_steps + timed_steps) * 0.1 + 30.0
    tabs = make_tables(args, n_envs, seed, horizon)
    cap = 384 if args.workload == "stress" else VEH_CAP
    orc = OracleScene(n_envs, cap, scene_params(vm=5 if args.workload == "stress" else VM), n_threads=n_threads)
    orc.reset(tabs, warmup=True)
    rng = np.random.RandomState(seed)

    def actions():
        if args.workload == "stress":
            return np.full((n_envs, cap), -3.0, np.float32)
        return rng.uniform(-3, 3, size=(n_envs, cap)).astype(np.float32)

    pool = [actions() for _ in range(8)]

    def masked(t):
        # the reference driver feeds 0 to uncontrolled vehicles (main.py:401-405); the CUDA arm does the same
        # through pve_config.zero_uncontrolled
        return np.where(orc.control_mask(), pool[t % 8], np.float32(0)).astype(np.float32)

    for t in range(prime + warmup_steps):
        orc.step(masked(t), reuse_buffers=True)
    agent_steps, veh_steps = 0, 0
    per_step = []
    for t in range(timed_steps):
        a = masked(t)                          # (not timed: the driver's side)
        t0 = time.perf_counter()
        o = orc.step(a, reuse_buffers=True)
        per_step.append(time.perf_counter() - t0)
        agent_steps += len(o["reward"])
    elapsed = float(sum(per_step))
    return {"agent_steps": agent_steps, "elapsed": elapsed, "n_envs": n_envs, "prime": prime, "threads": n_threads,
            "port": "oracle/scene_oracle.c (C port of the reference scene, persistent thread pool)"}


def cpu_port_run_lane4(args, n_envs, prime, timed_steps, warmup_steps, seed):
    """lane_num=4 / 8: the pure-Python oracles (oracle/scene4_oracle.py, scene8_oracle.py), one thread, a few intersections
    (the sample of intersections and the priming are bounded; every one of the `timed_steps` ticks is timed)."""
    from oracle.scene4_oracle import Scene4Oracle
    from oracle.scene8_oracle import Scene8Oracle
    n_envs, prime = min(n_envs, 4), min(prime, 200)
    tabs = make_tables(args, n_envs, seed, (prime + warmup_steps + timed_steps) * 0.1 + 30.0)
    if args.workload == "lane4":
        orcs = [Scene4Oracle(vm=VM) for _ in range(n_envs)]
        for o, t in zip(orcs, tabs):
            o.reset(t, warmup=True)
    else:
        orcs = [Scene8Oracle(vm=VM) for _ in range(n_envs)]
        draws = np.random.default_rng(0).integers(0, 2, size=tabs.shape, dtype=np.uint8)
        for o, t, d in zip(orcs, tabs, draws):
            o.reset(t, d, warmup=True)
    rng = np.random.RandomState(seed)
    agent_steps, elapsed = 0, 0.0
    for t in range(prime + warmup_steps + timed_steps):
        for o in orcs:
            m = np.array(o.control_mask(), bool)
            a = np.where(m, rng.uniform(-3, 3, size=len(m)), 0.0)
            t0 = time.perf_counter()
            out = o.step(a)
            if t >= prime + warmup_steps:
                elapsed += time.perf_counter() - t0
                agent_steps += len(out["ids"])
    return {"agent_steps": agent_steps, "elapsed": elapsed, "n_envs": n_envs, "prime": prime, "threads": 1,
            "port": "oracle/scene%d_oracle.py (Python port of the reference scene with lane_num=%d)" % ((lanes_of(args),) * 2)}


def reference_arm(args, rank):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n_envs = max(256, min(4096, 64 * cores))
    r = cpu_port_run(args, n_envs, PRIME_TICKS, args.steps, args.warmup, cores)
    value = r["agent_steps"] / r["elapsed"]
    sample = ("each step = one tick of %d intersections (bounded sample of the workload) on %d host threads, "
              "after %d priming ticks" % (r["n_envs"], r["threads"], r["prime"]))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * r["elapsed"] / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args), "reference_sample_envs": r["n_envs"],
                   "same_config": r["n_envs"] == args.envs,
                   "note": "agent-steps/s is a per-agent-step rate: the sample has the workload's density, actions and "
                           "occupancy but fewer intersections per step than the CUDA arm"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": r["threads"], "kind": "port", "sample": sample,
                         "python_reference": python_reference_rate(args)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)



# ---------------------------------------------------------------------------------------------
# the reference's own Python scene, when it is reachable (the build container); else its recorded rate
# ---------------------------------------------------------------------------------------------
REF_SCENE = "/root/reference/traffic_interaction_scene.py"
BASELINE_MD_PY_RATE = 6278.0       # BASELINE.md section 3: vehicle-agent env-steps/s on 1 core, density 1000, random actions


def _py_ref_worker(job):
    """One process = one independent TrafficInteraction driven like main.py:397-441 (random actions, 0 for uncontrolled)."""
    seed, density, warm, timed = job
    import argparse as _ap
    import types
    mpl, plt = types.ModuleType("matplotlib"), types.ModuleType("matplotlib.pyplot")
    mpl.pyplot = plt
    sys.modules.setdefault("matplotlib", mpl)
    sys.modules.setdefault("matplotlib.pyplot", plt)
    src = open(REF_SCENE, encoding="utf-8").read().split("\n")
    assert src[370].strip().startswith("for v in self.virtual_lane_4[0]:")
    for k in range(370, 375):                      # logging-only loop that raises IndexError (SURVEY.md Q9); output-neutral
        src[k] = "        pass"
    mod = types.ModuleType("ref_scene")
    exec(compile("\n".join(src), REF_SCENE, "exec"), mod.__dict__)
    from pve_mcc_for_unsignalized_intersection_b200.arrivals import synthetic_arrivals
    tab = synthetic_arrivals(1, density, (warm + timed) * 0.1 + 30.0, seed=seed)[0]
    env = mod.TrafficInteraction(tab, 150, _ap.Namespace(collision_thr=2, o_agent_num=6, c_mode="closer"), vm=VM, lane_num=12)
    rng = np.random.RandomState(seed)
    n, t0 = 0, 0.0
    for t in range(warm + timed):
        if t == warm:
            t0 = time.perf_counter()
        for lane in range(12):
            for ind, veh in enumerate(env.veh_info[lane]):
                env.step(lane, ind, float(rng.uniform(-3, 3)) if veh["control"] else 0)
        out = env.scene_update()
        env.delete_vehicle()
        if t >= warm:
            n += len(out[0])
    return n, time.perf_counter() - t0


def python_reference_rate(args):
    """agent-steps/s of the reference's own Python scene step on this host (all cores, one scene per process), when
    /root/reference is present; otherwise the rate BASELINE.md records for it, labelled as quoted."""
    if args.workload != "poisson":
        return None
    if not os.path.exists(REF_SCENE):
        return {"value_per_core": BASELINE_MD_PY_RATE, "unit": UNIT, "source": "quoted from BASELINE.md section 3 "
                "(reference scene, 1 core of the survey container; /root/reference does not exist on this host)"}
    try:
        import multiprocessing as mp
        cores = os.cpu_count() or 1
        with mp.get_context("fork").Pool(cores) as pool:
            res = pool.map(_py_ref_worker, [(4000 + i, args.density, 300, 200) for i in range(cores)])
        total = sum(n for n, _ in res)
        slowest = max(dt for _, dt in res)
        return {"value": total / slowest, "value_per_core": total / slowest / cores, "unit": UNIT, "cores": cores,
                "source": "measured now: %s under multiprocessing.Pool(%d), one scene per process, 300 warm-up + 200 "
                          "timed ticks each (main.py:397-441 loop)" % (REF_SCENE, cores)}
    except Exception as e:      # noqa: BLE001 - a reported baseline must never break the bench
        return {"value_per_core": BASELINE_MD_PY_RATE, "unit": UNIT, "source": "quoted from BASELINE.md section 3 (run failed: %r)" % (e,)}


# ---------------------------------------------------------------------------------------------
# DRAM traffic of one step-kernel launch, measured by a one-launch ncu child of this very script
# ---------------------------------------------------------------------------------------------
def traffic_child(args):
    """`bench.py --traffic-child`: the bench workload up to a few timed-like ticks; ncu profiles one of them."""
    import torch
    from pve_mcc_for_unsignalized_intersection_b200 import SceneConfig
    from pve_mcc_for_unsignalized_intersection_b200.scene import BatchedScene
    dev = torch.device("cuda", 0)
    B = args.envs
    stress = args.workload == "stress"
    veh_cap, agent_cap = (384, 320) if stress else (args.veh_cap, args.agent_cap)
    scene = BatchedScene(B, SceneConfig(vm=5 if stress else VM, zero_uncontrolled_actions=True,
                                        lane_num=lanes_of(args)), veh_cap=veh_cap,
                         agent_cap=agent_cap, device=dev, threads=args.threads)
    scene.reset(make_tables(args, B, 1000, (PRIME_TICKS + 60) * 0.1 + 30.0), warmup=True)
    gen = torch.Generator(device=dev)
    gen.manual_seed(99)
    pool = [(torch.full((B, veh_cap), -3.0, device=dev) if stress else
             (torch.rand(B, veh_cap, device=dev, generator=gen) * 6.0 - 3.0).contiguous()) for _ in range(4)]
    flush = torch.empty(384 * 1024 * 1024, dtype=torch.uint8, device=dev)
    for t in range(PRIME_TICKS + 8):
        if t >= PRIME_TICKS:
            flush.fill_(t & 0xFF)
        scene.step(pool[t % 4])
    torch.cuda.synchronize()


def measure_traffic(args, veh_cap, agent_cap):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the step kernel at this workload, from an ncu child
    (two metrics: a single replay pass).  Returns (bytes, how) or (None, why)."""
    import shutil
    import subprocess
    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    if not os.path.exists(ncu):
        return None, "ncu not found"
    # launches of pve_step_kernel before the profiled one: the reset's warm-up tick + PRIME_TICKS + 4 flushed ticks
    cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none", "-k",
           "regex:pve4_step_kernel" if lanes_of(args) != 12 else "regex:pve_step_kernel", "-s", str(PRIME_TICKS + 5), "-c", "1",
           "--csv", sys.executable,
           os.path.abspath(__file__), "--traffic-child", "--envs", str(args.envs), "--density", str(args.density),
           "--workload", args.workload, "--threads", str(args.threads), "--veh-cap", str(veh_cap),
           "--agent-cap", str(agent_cap)]
    try:
        res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=240)
    except Exception as e:      # noqa: BLE001
        return None, "ncu child failed: %r" % (e,)
    import csv
    import io
    tot, seen = 0.0, 0
    unit_scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith('"')]
    for row in csv.DictReader(io.StringIO("\n".join(lines))):
        if row.get("Metric Name") in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            try:
                tot += float(row["Metric Value"].replace(",", "")) * unit_scale.get(row.get("Metric Unit", "byte"), 1.0)
                seen += 1
            except ValueError:
                pass
    if seen != 2:
        return None, "ncu child gave no dram metrics (rc %d): %s" % (res.returncode, (res.stdout + res.stderr)[-300:].replace("\n", " | "))
    return tot, "measured in this run: ncu child, one launch of pve_step_kernel, dram__bytes_read.sum + dram__bytes_write.sum"


def committed_traffic():
    """The newest committed ncu capture of the step kernel, tagged with its file and commit (fallback only)."""
    import glob
    import subprocess
    caps = sorted(glob.glob(os.path.join(ROOT, "profiles", "*step_kernel*_full.json")))
    if not caps:
        return None, None
    try:
        val = json.load(open(caps[-1]))["derived"]["dram_traffic_bytes_per_launch"]
        sha = subprocess.run(["git", "-C", ROOT, "log", "-n", "1", "--format=%h", "--", caps[-1]], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                             text=True).stdout.strip() or None
        return val, {"source": os.path.relpath(caps[-1], ROOT), "commit": sha,
                     "note": "NOT measured in this run: value of a committed ncu capture of an earlier build"}
    except Exception:           # noqa: BLE001
        return None, None


# ---------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi equivalent through NVML), running during the timed region
# ---------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        while not self.stop_flag and self.nv is not None:
            try:
                self.sm.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.01)

    def result(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


# ---------------------------------------------------------------------------------------------
# --dump-outputs: what the last timed tick computed, for comparing two builds output for output
# ---------------------------------------------------------------------------------------------
DUMP_BYTES = 64 * 10**6          # decimal MB; sample_outputs leaves 1 MiB of it for the .npy headers


def last_outputs(scene, out, actions, folder):
    """name -> host array of what the last timed tick handed its caller: the step's outputs (``StepOutputs``: the
    reference's 9-tuple), in a rollout the policy's actions, in a training rollout the replay records its push
    appended.  None when the scene overflowed: that run is discarded and repeated in the next capacity class."""
    import torch
    if scene.stats()["overflow"]:
        return None
    n = out.n_agents
    got = {f: getattr(out, f) for f in ("agent_offset", "env_collisions", "env_lock", "env_removed")}
    got.update({f: getattr(out, f)[:n] for f in ("obs", "reward", "ids", "cpv", "status", "jerk_sum")})
    if actions is not None:
        got["actions"] = actions
    if folder is not None:
        c = folder.counters()
        pos = torch.arange(c["num_experiences"] - c["last_added"], c["num_experiences"], device=out.obs.device)
        got.update({"replay_" + k: v[pos % folder.capacity] for k, v in folder.arrays().items()})
    return sample_outputs({k: v.cpu().numpy() for k, v in got.items()})


def sample_outputs(arrays, budget=DUMP_BYTES - (1 << 20)):
    """float32 arrays stay float32, integer ones become float64 (exact).  Whatever does not fit ``budget`` bytes in
    all: the smallest arrays are kept whole, each larger one keeps an equal share of what is left as a seeded sample
    of its rows (``<name>_rows``: the row numbers, ascending).  Same shapes in, same rows out."""
    arrays = {k: v if v.dtype == np.float32 else v.astype(np.float64) for k, v in arrays.items()}
    out, left = {}, budget
    for i, name in enumerate(sorted(arrays, key=lambda k: (arrays[k].nbytes, k))):
        v, share = arrays[name], left // (len(arrays) - i)
        if v.nbytes <= share:
            out[name] = v
        else:
            keep = share // (v.nbytes // len(v) + 8)
            rows = np.sort(np.random.default_rng(0).permutation(len(v))[:keep])
            out[name], out[name + "_rows"] = v[rows], rows.astype(np.float64)
        left -= out[name].nbytes + (out[name + "_rows"].nbytes if name + "_rows" in out else 0)
    return out


# ---------------------------------------------------------------------------------------------
# the GPU arm
# ---------------------------------------------------------------------------------------------
def graft_arm(args, rank, world, local_rank, veh_cap, agent_cap):
    import torch
    import torch.distributed as dist
    from pve_mcc_for_unsignalized_intersection_b200 import SceneConfig
    from pve_mcc_for_unsignalized_intersection_b200.scene import BatchedScene

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the environment step has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # one rank per GPU on one host: give every rank its own cores (host threads of the pipelined host path and of the
        # launches do not migrate or compete) -- the node's GPUs all report the same CPU affinity, so a plain split
        try:
            cpus = sorted(os.sched_getaffinity(0))
            per = max(1, len(cpus) // world)
            mine = cpus[local_rank * per:(local_rank + 1) * per] or cpus
            os.sched_setaffinity(0, mine)
        except (AttributeError, OSError):
            pass
    if world > 1 and not dist.is_initialized():
        # stdout carries exactly one JSON line: whatever the communicator set-up writes to file descriptor 1 (NCCL's
        # banner and, with NCCL_DEBUG=INFO, its log) goes to stderr instead; NCCL_DEBUG itself is left as the caller set it
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)                  # creates the communicator now, not inside the timed region
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    B = args.envs
    K, W = args.steps, args.warmup
    stress = args.workload == "stress"
    horizon = (PRIME_TICKS + 5 * (K + W) + 50) * 0.1 + 30.0
    tabs = make_tables(args, B, 1000 + rank, horizon)
    rollout = args.workload in ("rollout", "train")
    # every slot of the action tensor is filled; the library takes the action of an uncontrolled vehicle as 0, which is
    # what the reference driver feeds (main.py:401-405)
    scene = BatchedScene(B, SceneConfig(vm=5 if (stress or rollout) else VM, zero_uncontrolled_actions=True,
                                        lane_num=lanes_of(args)),
                         veh_cap=veh_cap, agent_cap=agent_cap, device=dev, threads=args.threads,
                         neighbour_sources=args.workload == "train",
                         out_cap=B * args.out_rows_per_env if args.out_rows_per_env else None)
    scene.reset(tabs, warmup=True)
    actor = None
    if rollout:
        from pve_mcc_for_unsignalized_intersection_b200.actor import ActorWeights, BatchedActor
        actor = BatchedActor(ActorWeights.from_npz(os.path.join(ROOT, "tests", "golden", "actor_agent1.npz")), device=dev)
        act_buf = torch.empty(B, veh_cap, dtype=torch.float32, device=dev)
    folder = None
    if args.workload == "train":
        from pve_mcc_for_unsignalized_intersection_b200.nstep import BatchedCritic, CriticWeights, NStepFolder
        with np.load(os.path.join(ROOT, "tests", "golden", "nstep_nets.npz")) as z:
            t_actor = BatchedActor(ActorWeights({k[len("actor__"):].replace("__", "/"): z[k] for k in z.files
                                                 if k.startswith("actor__")}), device=dev)
            t_critic = BatchedCritic(CriticWeights({k[len("critic__"):].replace("__", "/"): z[k] for k in z.files
                                                    if k.startswith("critic__")}), device=dev)
        folder = NStepFolder(scene, t_actor, t_critic, seq_max_step=12, buffer_size=max(500000, scene.out_cap + 1))   # main.py:91, 212 (a tick must fit)
    gen = torch.Generator(device=dev)
    gen.manual_seed(99 + rank)
    if stress:
        pool = [torch.full((B, veh_cap), -3.0, device=dev) for _ in range(2)]
    else:
        pool = [(torch.rand(B, veh_cap, device=dev, generator=gen) * 6.0 - 3.0).contiguous() for _ in range(16)]
    flush = torch.empty(384 * 1024 * 1024, dtype=torch.uint8, device=dev)     # > 126 MB L2

    def actions(t):
        """The step's input: a pre-generated random tensor, or (rollout) the policy evaluated now."""
        if actor is not None:
            return actor.act(scene, out=act_buf)
        return pool[t % len(pool)]

    def tick(a):
        """One tick of the workload: the environment step and, for `train`, main.py:243-266 on its outputs."""
        if folder is not None:
            folder.bind_outputs()              # the step writes its observations straight into the folder's frame log
        out = scene.step(a)
        if folder is not None:
            folder.push(out, TRAIN_GAMMA)
        return out

    for t in range(PRIME_TICKS):
        tick(actions(t))
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident timing (value, roofline) ----------------
    # Every timed tick is bracketed by its own CUDA-event pair on the launching stream (the L2 flush
    # in between is not timed).  The same K ticks are timed twice over: once by bench.py's events
    # around the public step() call (-> value) and, inside the library, by events placed directly
    # around the step kernel (pve_set_profiling -> roofline.achieved).
    for t in range(W):
        flush.fill_(t & 0xFF)
        tick(actions(t))
    s0 = scene.stats()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    barrier()
    wall0 = time.perf_counter()
    out = None
    for t in range(K):                         # the K timed ticks -> value
        flush.fill_(t & 0xFF)                  # L2 flush between timed iterations (not timed)
        ev[t][0].record()
        out = tick(actions(t))
        ev[t][1].record()
    barrier()
    wall1 = time.perf_counter()
    # copied to the host now: the ticks below reuse the output buffers
    dumped = (last_outputs(scene, out, act_buf if actor is not None else None, folder)
              if args.dump_outputs and rank == 0 and out is not None else None)
    step_ms = [e0.elapsed_time(e1) for e0, e1 in ev]
    first_timed = 1 + PRIME_TICKS + W          # index of the first timed step since reset
    order_launches = sum(1 for t in range(first_timed, first_timed + K) if t % 32 == 0) if B >= 1024 else 0
    s1 = scene.stats()
    dA = s1["agent_steps"] - s0["agent_steps"]
    dV = s1["vehicle_steps"] - s0["vehicle_steps"]
    total_ms = float(sum(step_ms))
    # K more ticks with the library's own events directly around the step kernel -> roofline
    scene.set_profiling(True)
    kern_ms = []
    actor_ms = []
    aev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    fev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    fold_ms = []
    for t in range(K):
        flush.fill_(t & 0xFF)
        if actor is not None:                  # the policy kernel of this tick, timed on its own
            aev[0].record()
            a = actions(K + t)
            aev[1].record()
            if folder is not None:
                folder.bind_outputs()
            out = scene.step(a)
            if folder is not None:             # the folding of this tick, timed on its own
                fev[0].record()
                folder.push(out, TRAIN_GAMMA)
                fev[1].record()
        else:
            scene.step(actions(K + t))
        kern_ms.append(scene.kernel_ms()[0])   # waits for this tick's kernel
        if actor is not None:
            actor_ms.append(aev[0].elapsed_time(aev[1]))
        if folder is not None:
            torch.cuda.synchronize()
            fold_ms.append(fev[0].elapsed_time(fev[1]))
    scene.set_profiling(False)
    sampler.stop_flag = True
    s2 = scene.stats()
    kA = s2["agent_steps"] - s1["agent_steps"]
    kV = s2["vehicle_steps"] - s1["vehicle_steps"]
    total_kern_ms = float(sum(kern_ms))

    # ---------------- end-to-end through host buffers ----------------
    # e2e: the full 9-tuple reaches pinned host memory every tick (observations included: the reference driver reads
    # veh["state"] and buffers state_next on the host, main.py:234-245); e2e_no_obs: everything but the observations
    e2e = {}
    if not args.no_e2e and actor is None:
        pairs = scene.make_async_buffers()
        hact = [p.cpu().pin_memory() for p in pool[:4]]
        for name, with_obs in (("e2e_no_obs", False), ("e2e", True)):
            host_s = [0.0, 0.0]

            def run(n_ticks):
                rows = 0
                for t in range(n_ticks):
                    c0 = time.perf_counter()
                    scene.step_host_async(hact[t % len(hact)], pairs[t % 3], copy_obs=with_obs)
                    c1 = time.perf_counter()
                    if t >= 2:
                        rows += scene.host_wait()[0]          # tick t - 2 is in host memory; ticks t - 1 and t are under way
                    host_s[0] += c1 - c0
                    host_s[1] += time.perf_counter() - c1
                for _ in range(min(2, n_ticks)):
                    rows += scene.host_wait()[0]
                return rows
            run(max(3, W))
            barrier()
            t0 = time.perf_counter()
            n_rows = run(K)
            barrier()
            e2e_s = time.perf_counter() - t0
            d2h = n_rows / K * (16 + (OBS_BYTES if with_obs else 0)) + (B + 1) * 4 + 3 * B * 4
            e2e[name] = {"agent_steps": n_rows, "seconds": e2e_s, "h2d": B * veh_cap * 4, "d2h": d2h}
            print("%s: %.1f us per tick; host time in step_host_async %.1f us, in host_wait %.1f us (incl. warm-up ticks)" % (
                name, 1e6 * e2e_s / K, 1e6 * host_s[0] / (K + max(3, W)), 1e6 * host_s[1] / (K + max(3, W))), file=sys.stderr)

    # ---------------- reduce over ranks ----------------
    vec = torch.tensor([total_ms, total_kern_ms, e2e["e2e"]["seconds"] if e2e else 0.0,
                        e2e["e2e_no_obs"]["seconds"] if e2e else 0.0], dtype=torch.float64, device=dev)
    sums = torch.tensor([dA, dV, e2e["e2e"]["agent_steps"] if e2e else 0.0,
                         e2e["e2e_no_obs"]["agent_steps"] if e2e else 0.0], dtype=torch.float64, device=dev)
    counters = scene.stats_tensor().clone()
    if world > 1:
        dist.all_reduce(vec, op=dist.ReduceOp.MAX)         # slowest rank defines the time
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
        dist.all_reduce(counters, op=dist.ReduceOp.SUM)    # end-of-rollout statistics over NVLink
    total_ms, total_kern_ms, e2e_s, e2e_no_s = [float(x) for x in vec.tolist()]
    dA_all, dV_all, e2e_rows, e2e_no_rows = [float(x) for x in sums.tolist()]

    overflow = float(counters[12].item())
    if overflow > 0 and not os.environ.get("PVE_BENCH_ALLOW_OVERFLOW"):      # (the env knob is for kernel experiments only)
        # an intersection needed more slots than the capacity class holds and an arrival was deferred: that run deviates
        # from the reference, so it is never reported -- main() repeats the whole measurement with the next class
        scene.close()
        return False
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
        # per-GPU achieved bandwidth of the step kernel: this rank's algorithmic bytes / its kernel time.
        # DRAM bytes of one launch: measured now by a one-launch ncu child of this script (single GPU only), else the
        # value of the newest committed capture, tagged with its file and commit
        traffic, traffic_src = None, None
        if world == 1 and not args.no_traffic and args.workload in ("poisson", "stress", "lane4", "lane8"):
            traffic, traffic_src = measure_traffic(args, veh_cap, agent_cap)
        if traffic is None and args.envs == ENVS_PER_GPU and args.workload == "poisson":
            why = traffic_src
            traffic, traffic_src = committed_traffic()
            if traffic_src is not None and why:
                traffic_src["why_not_measured"] = why if world == 1 else "multi-GPU run: ncu is never wrapped around ranks"
        alg_bytes = BYTES_PER_VEH * kV + BYTES_PER_AGENT * kA
        my_kern_ms = float(sum(kern_ms))
        achieved = alg_bytes / (my_kern_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": dA_all / (total_ms * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": total_ms / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(args), "l2": "flushed between timed steps (384 MiB fill)",
                       "prime_ticks": PRIME_TICKS, "veh_cap": veh_cap, "agent_cap": agent_cap,
                       "threads_per_cta": scene.threads, "smem_per_cta": scene.smem_bytes,
                       "launch": scene.launch_info,
                       "agents_per_env_step": dA / (K * B), "vehicles_per_env_step": dV / (K * B),
                       "env_steps_per_s": world * B * K / (total_ms * 1e-3)},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_src,
                         "kernel": "pve4_step_kernel" if lanes_of(args) != 12 else "pve_step_kernel",
                         "kernel_ms_per_launch": my_kern_ms / K,
                         "algorithmic_bytes_per_launch": alg_bytes / K},
            # kernels inside the timed region of `value`: one step kernel per tick (+ one actor kernel in a rollout)
            # (+ target actor on this tick's rows and on last tick's referenced rows, mark, gather, critic, plan, scan,
            # fold in a training rollout; the memset of the marks is a driver operation)
            # + pve_order_kernel, launched by every 32nd step since reset (the warm-up tick inside reset is step 0)
            # per tick: the step (two concurrent kernels in dual mode; offsets + step + group sums on the 4-lane path), + the actor
            # kernel in a rollout, + target actor x 2, mark, gather, critic, plan, scan, fold in a training rollout
            "gpu_launches": (3 * K if lanes_of(args) != 12 else
                             K * ((2 if scene.launch_info["dual"] else 1) + (1 if actor is not None else 0) + (8 if folder is not None else 0))
                             + order_launches),
            "clocks": sampler.result(),
            "stats": {k: float(v) for k, v in zip(
                ["agent_steps", "vehicle_steps", "env_steps", "spawned", "passed", "passed_step_total",
                 "passed_jerk_sum", "collided_agent_steps", "lock_events", "reward_sum", "reward_sq_sum",
                 "removed", "overflow"], counters.tolist())},
            "wall_s_timed_region": wall1 - wall0,
        }
        if actor is not None:
            # 2 * (28*64 + 64*64 + 64) multiply-adds per agent; bytes: 112 B row in, 4 B action out, 8 B meta per slot
            line["actor"] = {"kernel": {"tc5": "pve_actor_tc_kernel", "mma": "pve_actor_mma_kernel", "ffma": "pve_actor_kernel"}.get(
                                 os.environ.get("PVE_ACTOR_IMPL", ""), "pve_actor_tc_kernel" if B * veh_cap >= 16384 else "pve_actor_mma_kernel"),
                             "kernel_ms_per_launch": float(sum(actor_ms)) / K,
                             "gflop_per_launch": 2 * 5952 * kA / K / 1e9,
                             "tflops": 2 * 5952 * kA / (float(sum(actor_ms)) * 1e-3) / 1e12,
                             "note": "tcgen05.mma + tensor memory (csrc/mlp_tc5.cuh), bf16 x 3 split-precision products "
                                     "(fp32-equivalent: the reference's "
                                     "graph is fp32 and ill-conditioned at 1e-4); tflops counts the network's fp32 "
                                     "multiply-adds once; timed alone with a cold L2, inside the same ticks as roofline"}
        if folder is not None:
            fc = folder.counters()
            # per agent row: 784 B observation in + 784 B frame out; per record: 2 x 784 B frames in, 2 x 784 + 36 B out
            fold_bytes = (1568 * kA + 3172 * kA) / K
            line["nstep"] = {"kernels": "pve_actor_tc_kernel x 2 (distinct rows: this tick's agents, last tick's referenced "
                                        "rows) + pvn_mark/gather + pve_critic_tc_kernel + pvn_plan/scan/fold",
                             "ms_per_push": float(sum(fold_ms)) / K, "seq_max_step": 12, "gamma": TRAIN_GAMMA,
                             "num_experiences": fc["num_experiences"], "records_last_push": fc["last_added"],
                             "slot_conflicts": fc["slot_conflicts"], "replay_capacity": folder.capacity,
                             "fold_algorithmic_bytes_per_push": fold_bytes,
                             "note": "timed alone with a cold L2 inside the same ticks as roofline; the bootstrap needs the "
                                     "target actor on all 7 rows of every agent's observation (main.py:253-255): it is "
                                     "evaluated once per distinct row and gathered through pve_outputs.nbr_src"}
        if e2e:
            line["e2e"] = {"value": e2e_rows / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(e2e["e2e"]["h2d"]),
                           "d2h_bytes_per_step": int(e2e["e2e"]["d2h"]),
                           "note": "pve_step_host_async + pve_host_wait, three ticks in flight: every tick's actions travel from pinned "
                                   "host memory (DMA) and the whole 9-tuple -- the 7x28 observation of every agent, a 16-byte record "
                                   "{reward, uid, lane, j, status, cpv, jerk_sum} per agent, offsets, per-intersection counters -- is "
                                   "in pinned host memory when pve_host_wait returns for that tick; ticks t+1 and t+2 are enqueued before "
                                   "tick t is waited for (the actions are pre-generated, as in the device-resident measurement)"}
            line["e2e_no_obs"] = {"value": e2e_no_rows / e2e_no_s, "unit": UNIT,
                                  "h2d_bytes_per_step": int(e2e["e2e_no_obs"]["h2d"]),
                                  "d2h_bytes_per_step": int(e2e["e2e_no_obs"]["d2h"]),
                                  "note": "as e2e, but the observations stay in HBM (a consumer whose policy runs on the device)"}
        if world == 1 and not args.no_cpu_baseline and actor is None:
            cores = os.cpu_count() or 1
            n_envs = max(256, min(2048, 32 * cores))
            r = cpu_port_run(args, n_envs, PRIME_TICKS, 100, 5, cores)
            r1 = cpu_port_run(args, 32, PRIME_TICKS, 100, 5, 1)
            line["cpu_baseline"] = {
                "value": r["agent_steps"] / r["elapsed"], "unit": UNIT, "cores": r["threads"], "kind": "port",
                "single_thread_value": r1["agent_steps"] / r1["elapsed"],
                "python_reference": python_reference_rate(args),
                "same_config": False,
                "sample": "%s: %d intersections x 100 ticks after %d priming ticks on %d threads (a per-agent-step rate "
                          "on a bounded sample of the workload, not the 4096-intersection batch); single-thread figure on "
                          "%d intersections" % (r["port"], r["n_envs"], r["prime"], r["threads"], r1["n_envs"])}
        if dumped is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in dumped.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
            print("dump-outputs: %d arrays, %.1f MB in %s" % (len(dumped), sum(a.nbytes for a in dumped.values()) / 1e6,
                                                             args.dump_outputs), file=sys.stderr)
        print(json.dumps(line), flush=True)
    return True


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        reference_arm(args, rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # plain `python bench.py --gpus N`: re-launch under torchrun, one rank per GPU
        import subprocess
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29531", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    if args.traffic_child:
        traffic_child(args)
        return
    # capacity classes, smallest first: a run that overflows its class is discarded and repeated with the next one
    classes = [(96, 48), (96, 64), (128, 80), (128, 96), (192, 128), (384, 320), (576, 416)]
    want = (384, 320) if args.workload == "stress" else (args.veh_cap, args.agent_cap)
    todo = [c for c in classes if c[0] >= want[0] and c[1] >= want[1]]
    if lanes_of(args) != 12:                   # the 4- / 8-lane path has two classes: 64/64 and 128/96
        todo = [(64, 64), (128, 96)] if args.workload == "lane4" and args.veh_cap == VEH_CAP else [(128, 96)]
    for vc, ac in todo:
        if graft_arm(args, rank, world, local_rank, vc, ac):
            break
    else:
        raise SystemExit("every capacity class overflowed: no valid measurement")
    if world > 1:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.barrier()
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
