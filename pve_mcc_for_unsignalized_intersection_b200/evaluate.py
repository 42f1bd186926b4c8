"""Evaluation of a pretrained policy on arrival-table files: the reference's ``--type test`` /
``batch_test`` drivers (main.py:367-441 and 543-583) on the GPU (SURVEY.md section 8(f), row N4).

The reference loops over seven density files, simulates 36 000 ticks of one intersection each with the
actor in the loop, and writes one line per file:

    vehicle number %s  collisions occurred number %s collisions rate %s pT-m %0.4f s jerks %s lock_num %s

Here all files run side by side as the intersections of one ``BatchedScene`` (each with its own table), the
actor is evaluated by ``BatchedActor``; the per-file tallies are kept on the device and read once at the end.
``format_report`` reproduces the line character by character from the same quantities.
"""
import os

import numpy as np
import torch

from . import _native as N
from .actor import ActorWeights, BatchedActor
from .config import NLANE, SceneConfig
from .scene import BatchedScene

DENSITIES = (1200, 1000, 900, 800, 600, 400, 200)              # main.py:545


def load_arrivals(mat_path):
    """``scipy.io.loadmat(mat_path)["arvTimeNewVeh"]`` (main.py:388-389, 551-552) as float64 ``[K, 12]``."""
    import scipy.io as scio
    arr = np.asarray(scio.loadmat(mat_path)["arvTimeNewVeh"], dtype=np.float64)
    if arr.ndim != 2 or arr.shape[1] != NLANE:
        raise ValueError("%s: arvTimeNewVeh has shape %s, expected [K, %d]" % (mat_path, arr.shape, NLANE))
    return arr


def stack_tables(tables):
    """Tables of different length -> one ``[B, K, 12]`` array, zero-padded (zeros = no more arrivals)."""
    K = max(t.shape[0] for t in tables)
    out = np.zeros((len(tables), K, NLANE), dtype=np.float64)
    for b, t in enumerate(tables):
        out[b, :t.shape[0]] = t
    return out


def format_report(vehicles, collisions, passed, passed_step_total, jerk_total, lock_total, deltaT=0.1):
    """The result line of main.py:576-581."""
    return ("vehicle number %s  collisions occurred number %s collisions rate %s pT-m %0.4f s jerks %s "
            "lock_num %s" % (vehicles, collisions, float(collisions) / vehicles,
                             float(passed_step_total) / (passed + 0.0001) * deltaT, jerk_total / passed, lock_total))


_TALLIES = ("vehicles", "collisions", "passed", "passed_step_total", "jerk_total", "lock_total")   # format_report's


def evaluate_tables(tables, weights, ticks=36000, vm=5, collision_thr=2, device="cuda:0", veh_cap=128,
                    agent_cap=96, progress=None):
    """Closed loop actor + scene on every table of ``tables`` (list of ``[K, 12]`` arrays) for ``ticks``
    ticks.  Returns one dict per table with the quantities of main.py:566-581."""
    return _evaluate(len(tables), lambda scene: scene.reset(stack_tables(tables), warmup=True), weights, ticks, vm,
                     collision_thr, device, veh_cap, agent_cap, progress)


def evaluate_poisson(weights, densities=DENSITIES, envs_per_density=64, ticks=36000, seed=0, min_headway=1.0, vm=5,
                     collision_thr=2, device="cuda:0", veh_cap=192, agent_cap=128, progress=None):
    """The density sweep of ``batch_test`` on generated traffic: ``envs_per_density`` intersections per density (veh/h
    and lane), all of one density contiguous, in one scene with one ``reset_poisson`` of per-intersection rates, the
    closed loop of ``evaluate_tables`` for ``ticks`` ticks.  Returns one dict per density: ``"density"``,
    ``"intersections"`` (the dicts ``evaluate_tables`` returns, one per intersection), ``"pooled"`` (their sums) and
    ``"report"`` (``format_report`` of the pooled sums)."""
    n = int(envs_per_density)
    rates = np.repeat(np.asarray(densities, dtype=np.float64), n)[:, None]
    res = _evaluate(len(rates), lambda scene: scene.reset_poisson(rates, seed, min_headway=min_headway, warmup=True),
                    weights, ticks, vm, collision_thr, device, veh_cap, agent_cap, progress)
    out = []
    for k, d in enumerate(densities):
        per = res[k * n:(k + 1) * n]
        pooled = {q: sum(r[q] for r in per) for q in _TALLIES}
        out.append({"density": d, "intersections": per, "pooled": pooled, "report": format_report(**pooled)})
    return out


def _evaluate(B, reset, weights, ticks, vm, collision_thr, device, veh_cap, agent_cap, progress):
    """``reset(scene)`` on a new scene of ``B`` intersections, then the closed loop; one dict of tallies per
    intersection."""
    scene = BatchedScene(B, SceneConfig(vm=vm, collision_thr=collision_thr), veh_cap=veh_cap, agent_cap=agent_cap,
                         device=device)
    actor = BatchedActor(weights, device=device)
    reset(scene)
    dev = scene.device
    acts = torch.empty(B, scene.veh_cap, dtype=torch.float32, device=dev)
    # the tallies of main.py:567-571 (jerks of finished vehicles, lock events, agents with collision > 0) are kept per
    # intersection by the step kernel itself (pve_env_stats_dev): the loop is enqueued by the library (pve_rollout, 1000
    # ticks per call) and never synchronises; the sticky overflow counter is looked at every 2000 ticks so that a run that left the capacity class
    # stops early
    done = 0
    while done < ticks:
        n = min(1000, ticks - done)
        actor.rollout(scene, n, out=acts)                            # main.py:557-566 (+ delete_vehicle, 575), n ticks
        done += n
        if done % 2000 == 0 and scene.stats()["overflow"] != 0:
            break
        if progress:
            progress(done - 1, scene)
    es = scene.env_stats().cpu().numpy()
    names = list(scene.ENV_STAT_NAMES)
    coll = es[:, names.index("collided_agent_steps")]
    lock = es[:, names.index("lock_events")]
    jerk = es[:, names.index("passed_jerk_sum")]
    st = scene.get_state()
    if int(st["overflow"].sum()) != 0:
        raise N.NativeError("capacity class %d/%d overflowed during the evaluation; rerun with larger caps"
                            % (scene.veh_cap, scene.agent_cap))
    res = []
    for b in range(B):
        res.append({"vehicles": int(st["id_seq"][b]), "collisions": int(coll[b]), "passed": int(st["passed_veh"][b]),
                    "passed_step_total": int(st["passed_step_total"][b]), "jerk_total": float(jerk[b]),
                    "lock_total": int(lock[b])})
        res[-1]["report"] = format_report(res[-1]["vehicles"], res[-1]["collisions"], res[-1]["passed"],
                                          res[-1]["passed_step_total"], res[-1]["jerk_total"], res[-1]["lock_total"])
    return res


def batch_test(model_dir, data_dir, out_path=None, densities=DENSITIES, lane_num=12, ticks=36000, device="cuda:0",
               veh_cap=192, agent_cap=128):
    """main.py:543-583: every ``arvTimeNewVeh_new_<density>_<lane_num>.mat`` of ``data_dir`` with the checkpoint
    of ``model_dir``; writes the reference's ``*_batch_test_result_12_v1.txt`` lines to ``out_path``."""
    if lane_num != NLANE:
        raise NotImplementedError("batch_test evaluates the shipped 12-lane checkpoint on the 12-lane arrival files (the "
                                  "reference ships neither for lane_num 4 / 8); use BatchedScene(SceneConfig(lane_num=...)) directly")
    weights = ActorWeights.from_checkpoint(model_dir)
    names = ["arvTimeNewVeh_new_%s_%s.mat" % (d, lane_num) for d in densities]
    tables = [load_arrivals(os.path.join(data_dir, n)) for n in names]
    res = evaluate_tables(tables, weights, ticks=ticks, device=device, veh_cap=veh_cap, agent_cap=agent_cap)
    lines = []
    for n, r in zip(names, res):
        lines.append(os.path.join("./data/test", n))                 # main.py:549-550
        lines.append(r["report"])
    if out_path:
        with open(out_path, "w") as f:
            f.write("\n".join(lines) + "\n")
    return res, lines
