"""n-step return folding and the replay memory on the GPU (SURVEY.md section 8(f), row N2).

The reference's training loop keeps, per vehicle, a Python list of transitions and folds it after every
``scene_update`` (main.py:243-266):

    veh["buffer"].append([state_now[seq], actions[seq], reward[seq], state_next[seq], veh["Done"]])
    if veh["Done"] or veh["count"] > seq_max_step:
        r_target = reward of the last transition (+ gamma * Q'(s', mu'(s'), mu'(neighbours)) unless Done)
        for cur_data in reversed(seq_data[:-1]): r_target = cur_data[2] + args.gamma * r_target
        agent1_memory_seq.add(state, action, r_target, state_next, False) of the OLDEST transition
        veh["buffer"].pop(0); veh["count"] -= 1

``NStepFolder.push(outputs, gamma)`` does this for every agent row of a ``BatchedScene.step`` at once and
appends the records to a device-resident replay memory with the semantics of the reference's
``ReplayBuffer(..., rand_s=True)`` (replay_buffer.py:8-9, 45-53; main.py:212).  ``BatchedCritic`` is
``agent_ddpg_target.Q`` (model_agent_maddpg.py:52-76, 123-125).

Kernels: ``csrc/nstep.cuh`` behind ``pve_critic_* / pve_nstep_*`` (include/pve_mcc.h).  No CPU fallback.
The prioritised ``rank_based.Experience`` memory (``rand_s=False``) is not used by main.py and is out of scope.
"""
import ctypes as C
import random

import numpy as np
import torch

from . import _native as N
from .checkpoint import latest_checkpoint, read_bundle
from .config import OBS_H, OBS_W

# variable names below the critic's scope (NET:52-76), in the order of the flat vector of include/pve_mcc.h
CRITIC_SPECS = (
    ("LayerNorm/gamma", (28,)), ("LayerNorm/beta", (28,)),
    ("dense/kernel", (28, 64)), ("dense/bias", (64,)),
    ("LayerNorm_1/gamma", (64,)), ("LayerNorm_1/beta", (64,)),
    ("dense_1/kernel", (71, 64)), ("dense_1/bias", (64,)),
    ("LayerNorm_2/gamma", (64,)), ("LayerNorm_2/beta", (64,)),
    ("dense_2/kernel", (64, 1)), ("dense_2/bias", (1,)),
)
CRITIC_FLOATS = sum(int(np.prod(s)) for _, s in CRITIC_SPECS)      # 6841


class CriticWeights:
    """The twelve tensors of one critic network, float32, keyed by the names of CRITIC_SPECS."""

    def __init__(self, tensors):
        self.tensors = {}
        for name, shape in CRITIC_SPECS:
            if name not in tensors:
                raise KeyError("critic tensor %s is missing" % name)
            arr = np.asarray(tensors[name], dtype=np.float32)
            if arr.shape != shape:
                raise ValueError("critic tensor %s has shape %s, expected %s" % (name, arr.shape, shape))
            self.tensors[name] = np.ascontiguousarray(arr)

    @classmethod
    def from_checkpoint(cls, prefix_or_dir, scope="agent1_target_critic"):
        """``scope``: ``agent1_critic`` (MADDPG('agent1'), main.py:200) or ``agent1_target_critic`` (main.py:201)."""
        import os
        prefix = latest_checkpoint(prefix_or_dir) if os.path.isdir(prefix_or_dir) else prefix_or_dir
        got = read_bundle(prefix, ["%s/%s" % (scope, n) for n, _ in CRITIC_SPECS])
        return cls({n: got["%s/%s" % (scope, n)] for n, _ in CRITIC_SPECS})

    @classmethod
    def random(cls, seed=0):
        """The reference's initialisation (NET:60-73: kernels U(-3e-3, 3e-3), LN gamma 1 / beta 0, biases 0)."""
        rng = np.random.default_rng(seed)
        t = {}
        for name, shape in CRITIC_SPECS:
            if name.endswith("kernel"):
                t[name] = rng.uniform(-3e-3, 3e-3, shape).astype(np.float32)
            elif name.endswith("gamma"):
                t[name] = np.ones(shape, np.float32)
            else:
                t[name] = np.zeros(shape, np.float32)
        return cls(t)

    def flat(self):
        out = np.concatenate([self.tensors[n].reshape(-1) for n, _ in CRITIC_SPECS]).astype(np.float32)
        assert out.size == CRITIC_FLOATS
        return out


def _cuda_device(device):
    device = torch.device(device)
    if device.type != "cuda" or not torch.cuda.is_available():
        raise N.NativeError("the n-step / critic kernels need a CUDA device (there is no CPU fallback)")
    return device


class BatchedCritic:
    """Device copy of one critic network (``agent.Q``, NET:123-125)."""

    def __init__(self, weights, device="cuda:0", _library=None):
        self.device = _cuda_device(device)
        self.lib = N.load_library(_library)
        self.weights = weights
        flat = weights.flat()
        self._h = C.c_void_p()
        rc = self.lib.pve_critic_create(flat.ctypes.data_as(C.c_void_p), flat.size, self.device.index or 0, C.byref(self._h))
        if rc != 0:
            raise N.NativeError("pve_critic_create failed with %d" % rc)

    def close(self):
        if getattr(self, "_h", None):
            self.lib.pve_critic_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def forward(self, obs, actions7, out=None):
        """``obs`` float32 ``[n, 7, 28]`` (row 0 is the critic's state input, main.py:257), ``actions7`` ``[n, 7]`` =
        ``[action, other_action...]`` (NET:81-83)  ->  Q ``[n]``."""
        if obs.device != self.device or obs.dtype != torch.float32 or obs.dim() != 3 or tuple(obs.shape[1:]) != (OBS_H, OBS_W):
            raise ValueError("obs must be a float32 [n, 7, 28] tensor on %s" % self.device)
        if actions7.device != self.device or actions7.dtype != torch.float32 or tuple(actions7.shape) != (obs.shape[0], OBS_H):
            raise ValueError("actions7 must be a float32 [n, 7] tensor on %s" % self.device)
        obs, actions7 = obs.contiguous(), actions7.contiguous()
        if out is None:
            out = torch.empty(obs.shape[0], dtype=torch.float32, device=self.device)
        stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        rc = self.lib.pve_critic_forward(self._h, obs.data_ptr(), actions7.data_ptr(), obs.shape[0], None, out.data_ptr(), stream)
        if rc != 0:
            raise N.NativeError("pve_critic_forward failed with %d" % rc)
        return out


class NStepFolder:
    """Per-vehicle transition buffers + replay memory of the training loop, for one ``BatchedScene``.

    ``seq_max_step`` = ``args.seq_max_step`` (main.py:91); ``buffer_size`` = first argument of ``ReplayBuffer``
    (main.py:212).  ``uid_slots``: history slots per intersection (power of two; default twice the vehicle capacity).

    ``factored``: keep the frame log in the factored form (``pve_nstep_create_factored``: row 0, previous row 0 and 8 row
    codes per agent, 240 instead of 784 bytes; ``log_bytes`` tells the size) and push from the factored observation.  The
    scene must export it (``BatchedScene(factored_obs=True)``, with or without ``full_obs``; 12-lane intersections only).
    The replay memory, counters and bootstrap values are those of a full-frame folder fed the same ticks, bit for bit.
    """

    factored = False

    def __init__(self, scene, target_actor, target_critic, seq_max_step=12, buffer_size=500000, uid_slots=None,
                 factored=False):
        self.device = _cuda_device(scene.device)
        self.lib = scene.lib
        self.scene, self.target_actor, self.target_critic = scene, target_actor, target_critic
        self.factored = bool(factored)
        if self.factored and getattr(scene.out, "obs_src", None) is None:
            raise ValueError("NStepFolder(factored=True) pushes the factored observation, and this scene does not export it: "
                             "create the scene with BatchedScene(factored_obs=True) (12-lane intersections only)")
        if uid_slots is None:
            uid_slots = 1 << int(np.ceil(np.log2(max(16, 2 * scene.veh_cap))))
        self.seq_max_step, self.buffer_size, self.uid_slots = int(seq_max_step), int(buffer_size), int(uid_slots)
        self._h = C.c_void_p()
        create = self.lib.pve_nstep_create_factored if self.factored else self.lib.pve_nstep_create
        rc = create(scene.B, self.uid_slots, self.seq_max_step, scene.out_cap, self.buffer_size,
                    self.device.index or 0, C.byref(self._h))
        if rc != 0:
            raise N.NativeError("pve_nstep_create failed with %d (seq_max_step <= 14, uid_slots a power of two >= 16, "
                                "buffer_size - 1 >= out_cap = %d)" % (rc, scene.out_cap))
        self.log_bytes = int(self.lib.pve_nstep_log_bytes(self._h))     # the frame log of the last seq_max_step + 2 pushes
        view = N.PveReplayView()
        self.lib.pve_nstep_replay(self._h, C.byref(view))
        self.capacity = int(view.capacity)                        # buffer_size - 1 (replay_buffer.py:47-53)
        self._view = view
        self._tensors = None

    def close(self):
        if getattr(self, "_h", None):
            self._tensors = None
            self.lib.pve_nstep_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def push(self, outputs, gamma, distinct_rows=None):
        """main.py:243-266 for the tick that produced ``outputs`` (a ``StepOutputs``).  Asynchronous.
        ``distinct_rows``: None = use the scene's neighbour sources when it exports them (``BatchedScene(
        neighbour_sources=True)``, any ``lane_num``); False = always evaluate the target actor on all 7 rows of every
        observation.  With neighbour sources the push reads the rows the step read, so it must come before the scene's
        next step.

        A factored folder reads the factored observation of ``outputs`` (any ``StepOutputs`` with ``row0_out``,
        ``prev_row0`` and ``obs_src``, not only ``scene.out``; ``obs`` is never read) and evaluates the target actor once
        per distinct row.  Its outputs carry every row the push needs, so the push may come after the scene's next step
        (give that step other outputs); pushes must still come in tick order."""
        if self.factored:
            if any(getattr(outputs, f, None) is None for f in ("row0_out", "prev_row0", "obs_src")):
                raise ValueError("a factored NStepFolder pushes the factored observation, and these outputs carry none "
                                 "(BatchedScene(factored_obs=True))")
            rc = self.lib.pve_nstep_push_factored(self._h, C.byref(outputs.native()), float(gamma), self.target_actor._h,
                                                  self.target_critic._h, self._stream())
            if rc != 0:
                raise N.NativeError("pve_nstep_push_factored failed with %d: %s"
                                    % (rc, self.lib.pve_nstep_last_error(self._h).decode()))
            return
        if outputs.obs is None:
            raise ValueError("NStepFolder.push reads the observations, and these outputs carry none (BatchedScene("
                             "full_obs=False)): call bind_outputs() before the step so that it writes them into the frame log")
        o = outputs.native()
        if distinct_rows is None:
            distinct_rows = getattr(outputs, "nbr_src", None) is not None and outputs is self.scene.out
        if distinct_rows:
            # the scene exported where every observation row came from (BatchedScene(neighbour_sources=True)): the
            # target actor runs once per distinct row instead of on all 7 rows of every agent (same results)
            rc = self.lib.pve_nstep_push_scene(self._h, self.scene._h, C.byref(o), float(gamma), self.target_actor._h,
                                               self.target_critic._h, self._stream())
        else:
            rc = self.lib.pve_nstep_push(self._h, C.byref(o), float(gamma), self.target_actor._h, self.target_critic._h,
                                         self._stream())
        if rc != 0:
            raise N.NativeError("pve_nstep_push failed with %d" % rc)

    def bind_outputs(self, outputs=None):
        """Zero-copy: make the next ``scene.step`` write its observations straight into the folder's frame log.  Call it
        before every step whose outputs will be pushed (``outputs`` defaults to ``scene.out``; its ``obs`` tensor is
        replaced by a view of the log block the next push expects, so read ``outputs.obs`` before the next call).
        Without it ``push`` copies the observation block into the log (same results, one more device copy per tick).
        A factored folder replaces ``row0_out``, ``prev_row0`` and ``obs_src`` instead (``pve_nstep_factored_slot``)."""
        outputs = self.scene.out if outputs is None else outputs
        if self.factored:
            ptrs = [C.c_void_p() for _ in range(3)]
            rc = self.lib.pve_nstep_factored_slot(self._h, *[C.byref(p) for p in ptrs])
            if rc != 0:
                raise N.NativeError("pve_nstep_factored_slot failed with %d" % rc)
            oc = self.scene.out_cap
            shapes = ((oc, OBS_W, torch.float32), (oc, OBS_W, torch.float32), (oc, 8, torch.int16))
            for name, p, (n, w, dt) in zip(("row0_out", "prev_row0", "obs_src"), ptrs, shapes):
                setattr(outputs, name, self._wrap(p.value, (n, w), dt))
                if outputs is self.scene.out:
                    setattr(self.scene._out_native, name, p.value)     # the struct the scene hands to pve_step
            return outputs
        ptr = C.c_void_p()
        rc = self.lib.pve_nstep_obs_slot(self._h, C.byref(ptr))
        if rc != 0:
            raise N.NativeError("pve_nstep_obs_slot failed with %d" % rc)
        outputs.obs = self._wrap(ptr.value, (self.scene.out_cap, OBS_H, OBS_W), torch.float32)
        if outputs is self.scene.out:
            self.scene._out_native.obs = ptr.value            # the struct the scene hands to pve_step
        return outputs

    def reset(self):
        """A new episode (main.py:230: a new ``TrafficInteraction`` per epoch): the vehicles' buffered transitions are
        dropped; the replay memory stays (``agent1_memory_seq`` is created once, main.py:212)."""
        rc = self.lib.pve_nstep_reset(self._h, self._stream())
        if rc != 0:
            raise N.NativeError("pve_nstep_reset failed with %d" % rc)

    def counters(self):
        """``num_experiences`` (replay_buffer.py:47), records added by the last push, history-slot conflicts, pushes.
        Synchronises.  Raises if a slot conflict was ever counted (``__len__``, ``order``, ``deque`` and ``get_batch`` go
        through here, so a corrupted memory cannot be read silently)."""
        out = (C.c_int64 * 4)()
        rc = self.lib.pve_nstep_counters(self._h, out, self._stream())
        if rc != 0:
            raise N.NativeError("pve_nstep_counters failed with %d" % rc)
        if int(out[2]) != 0:
            # two live vehicles of one intersection shared a history slot (uid mod uid_slots): their histories, and the
            # replay records folded from them, are no longer the reference's -- never hand such a memory out
            raise N.NativeError("n-step history table too small: %d slot conflicts (uid_slots must exceed the number of "
                                "vehicles an intersection spawns during one agent's lifetime); create the folder with a "
                                "larger uid_slots" % int(out[2]))
        if self.scene.stats()["overflow"] != 0:
            # an intersection outgrew its capacity class or the outputs did not fit out_cap: that tick's rows of the
            # intersection were not emitted (ADVICE r01), so transitions folded from them are not the reference's
            raise N.NativeError("the scene's sticky overflow counter is set (capacity class %d/%d or out_cap %d too small): "
                                "the replay memory may hold transitions of ticks whose rows were not emitted"
                                % (self.scene.veh_cap, self.scene.agent_cap, self.scene.out_cap))
        return {"num_experiences": int(out[0]), "last_added": int(out[1]), "slot_conflicts": int(out[2]), "pushes": int(out[3])}

    def __len__(self):
        """``len(memory.buffer)``"""
        return min(self.counters()["num_experiences"], self.capacity)

    def _wrap(self, ptr, shape, dtype):
        """Zero-copy tensor over library-owned device memory (CUDA array interface)."""
        class _Mem:
            pass
        m = _Mem()
        m.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": {torch.float32: "<f4", torch.uint8: "|u1", torch.int16: "<i2"}[dtype],
                                      "data": (int(ptr), False), "version": 2}
        return torch.as_tensor(m, device=self.device)

    def arrays(self):
        """The replay ring as tensors over the library's device memory (physical order, see ``order``)."""
        if self._tensors is None:
            c, v = self.capacity, self._view
            self._tensors = {
                "state": self._wrap(v.state, (c, OBS_H, OBS_W), torch.float32),
                "action": self._wrap(v.action, (c, OBS_H), torch.float32),
                "reward": self._wrap(v.reward, (c,), torch.float32),
                "next_state": self._wrap(v.next_state, (c, OBS_H, OBS_W), torch.float32),
                "done": self._wrap(v.done, (c,), torch.uint8),
            }
        return self._tensors

    def order(self):
        """Physical positions of the deque's items, oldest first (``list(memory.buffer)``)."""
        n = self.counters()["num_experiences"]
        first = max(0, n - self.capacity)
        return (torch.arange(first, n, device=self.device) % self.capacity)

    def deque(self):
        """The memory in the reference's order as a dict of tensors (copies)."""
        idx = self.order()
        return {k: t.index_select(0, idx) for k, t in self.arrays().items()}

    def get_batch(self, batch_size, rng=random):
        """``ReplayBuffer.getBatch`` with rand_s=True: ``random.sample(self.buffer, batch_size)`` (replay_buffer.py:20-22).
        Draws the same positions as the reference for the same ``random`` state."""
        idx = self.order()
        pick = torch.as_tensor(rng.sample(range(idx.numel()), batch_size), device=self.device, dtype=torch.long)
        phys = idx.index_select(0, pick)
        return {k: t.index_select(0, phys) for k, t in self.arrays().items()}

    def bootstrap_values(self):
        """Q' of the last push for its agent rows (diagnostics / tests)."""
        ptr = self.lib.pve_nstep_q_dev(self._h)
        return self._wrap(ptr, (self.scene.out_cap,), torch.float32)
