"""Host-side mirror of the reference scene for B independent intersections on one GPU.

``BatchedScene`` keeps the reference's reset/step contract (traffic_interaction_scene.py:
constructor 21-220, ``step`` 1501, ``scene_update`` 222, ``delete_vehicle`` 435): per-vehicle
accelerations in, per-agent observations / rewards / done flags / collision info out.  All
compute happens in the hand-written sm_100a kernels of ``csrc/`` behind the C ABI of
``include/pve_mcc.h``; torch tensors are used only as device buffers and for streams.
"""
import ctypes as C
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

from . import _native as N
from .arrivals import lane_rates, to_spawn_ticks
from .config import NLANE, OBS_H, OBS_W, SceneConfig


class StepOutputs:
    """Dense per-agent outputs of one tick (the reference's 9-tuple, TIS:376).

    Rows of intersection ``b`` are ``agent_offset[b]:agent_offset[b+1]`` in the reference's
    order (lane ascending, j ascending).  All tensors live on the scene's device; they are
    reused by the next ``step`` call.
    """

    def __init__(self, B, out_cap, device, neighbour_sources=False, records_only=False, factored=False, full_obs=True,
                 lib=None):
        z = lambda *s, dt: torch.zeros(*s, dtype=dt, device=device)
        e = lambda *s, dt: None
        per_agent = e if records_only else z                       # records_only: the 16-byte records replace them
        self.B, self.out_cap, self._lib = B, out_cap, lib
        # agent_offset and the three per-intersection counters share one allocation (one DMA on the host path)
        self._small = z(4 * B + 1, dt=torch.int32)
        self.agent_offset = self._small[:B + 1]
        # re_state; None with full_obs=False: the step does not write the 7 x 28 block at all
        self.obs = z(out_cap, OBS_H, OBS_W, dt=torch.float32) if full_obs else None
        self.reward = per_agent(out_cap, dt=torch.float32)
        self.ids = per_agent(out_cap, 4, dt=torch.int32)           # env, lane, j, uid
        self.cpv = per_agent(out_cap, dt=torch.int32)              # collisions_per_veh[:, 0]
        self.status = per_agent(out_cap, dt=torch.uint8)           # ST_DONE | ST_REMOVED | ST_FINISHED
        self.jerk_sum = per_agent(out_cap, dt=torch.float32)
        self.env_collisions = self._small[B + 1:2 * B + 1]         # `collisions`
        self.env_lock = self._small[2 * B + 1:3 * B + 1]           # `lock`
        self.env_removed = self._small[3 * B + 1:4 * B + 1]
        # pve_agent_record[out_cap]: reward, uid, lane, j, status, cpv, jerk_sum of a row in 16 bytes (the host path)
        self.packed = z(out_cap, 4, dt=torch.int32) if records_only else None
        # optional: where each of the 7 observation rows was copied from (include/pve_mcc.h, pve_outputs.nbr_src):
        # -1 zero row; g' = row 0 of agent g' of the same intersection this tick; 0x4000 | k = last tick's row of slot k
        # (BatchedScene.row0_prev).  Written by every lane_num (12, 8, 4).
        self.nbr_src = z(out_cap, 8, dt=torch.int16) if neighbour_sources else None
        # optional: the factored observation (include/pve_mcc.h, pve_outputs.row0_out / prev_row0 / obs_src): this tick's
        # row 0 of every agent, the row stored for its vehicle when the tick started, and per observation row a code:
        # -1 zero row, g' = row0_out of agent g' of the same intersection, 0x4000 | g' = prev_row0 of agent g'
        self.row0_out = z(out_cap, OBS_W, dt=torch.float32) if factored else None
        self.prev_row0 = z(out_cap, OBS_W, dt=torch.float32) if factored else None
        self.obs_src = z(out_cap, 8, dt=torch.int16) if factored else None
        self._n = None

    FIELDS = ("agent_offset", "obs", "reward", "ids", "cpv", "status", "jerk_sum",
              "env_collisions", "env_lock", "env_removed")

    def pin(self):
        """Move the (CPU) buffers to pinned memory, keeping agent_offset / env_* in one allocation."""
        B = self.env_lock.shape[0]
        self._small = self._small.pin_memory()
        self.agent_offset = self._small[:B + 1]
        self.env_collisions = self._small[B + 1:2 * B + 1]
        self.env_lock = self._small[2 * B + 1:3 * B + 1]
        self.env_removed = self._small[3 * B + 1:4 * B + 1]
        for f in ("obs", "reward", "ids", "cpv", "status", "jerk_sum", "packed", "row0_out", "prev_row0", "obs_src"):
            if getattr(self, f) is not None:
                setattr(self, f, getattr(self, f).pin_memory())
        return self

    def native(self):
        o = N.PveOutputs()
        for f in self.FIELDS:
            t = getattr(self, f)
            setattr(o, f, t.data_ptr() if t is not None else None)
        o.nbr_src = self.nbr_src.data_ptr() if self.nbr_src is not None else None
        o.packed = self.packed.data_ptr() if self.packed is not None else None
        for f in ("row0_out", "prev_row0", "obs_src"):
            t = getattr(self, f)
            setattr(o, f, t.data_ptr() if t is not None else None)
        return o

    def expand_obs(self, n=None, out=None, threads=1):
        """The observations ``[n, 7, 28]`` rebuilt bit for bit from the factored block (``row0_out``, ``prev_row0``,
        ``obs_src``), into ``out`` (float32 ``[>= n, 7, 28]`` on the buffers' device, allocated if None); returns
        ``out[:n]``.  ``n`` defaults to this tick's row count.  Device buffers: one kernel on the current stream
        (``pve_expand_obs``).  Host buffers: the C expander (``pve_expand_obs_host``) over ``threads`` ranges of
        intersections in parallel (the calls release the GIL).  Raises ``ValueError`` if a code is out of range."""
        if self.obs_src is None:
            raise ValueError("these outputs carry no factored observation (BatchedScene(factored_obs=True), "
                             "make_async_buffers(factored=True))")
        lib = self._lib or N.load_library()
        dev = self.obs_src.device
        n = self.n_agents if n is None else int(n)
        if out is None:
            out = torch.empty(max(n, 1), OBS_H, OBS_W, dtype=torch.float32, device=dev)
        if (out.dtype != torch.float32 or out.device != dev or not out.is_contiguous() or out.dim() != 3
                or tuple(out.shape[1:]) != (OBS_H, OBS_W) or out.shape[0] < n):
            raise ValueError("out must be a contiguous float32 [>= %d, 7, 28] tensor on %s" % (n, dev))
        # rows past n (and past the buffers) are never touched: the expanders skip intersections beyond the cap
        cap = min(n, self.row0_out.shape[0], self.prev_row0.shape[0], self.obs_src.shape[0])
        ptrs = (self.row0_out.data_ptr(), self.prev_row0.data_ptr(), self.obs_src.data_ptr(), out.data_ptr())
        if dev.type == "cuda":
            stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            rc = lib.pve_expand_obs(self.agent_offset.data_ptr(), self.B, cap, *ptrs, stream)
            if rc != 0:
                raise N.NativeError("pve_expand_obs failed with %d" % rc)
            return out[:n]
        off = self.agent_offset.numpy()
        bounds = [0, self.B]
        if threads > 1 and self.B > 1:      # ranges of about equal row counts
            cuts = np.searchsorted(off[:self.B + 1], np.arange(1, threads) * (n / threads), side="left")
            bounds = sorted(set([0, self.B] + [int(min(max(c, 0), self.B)) for c in cuts]))
        ranges = list(zip(bounds[:-1], bounds[1:]))
        call = lambda r: int(lib.pve_expand_obs_host(self.agent_offset.data_ptr(), r[0], r[1], cap, *ptrs))
        if len(ranges) == 1:
            bad = [call(ranges[0])]
        else:
            bad = list(_pool(threads).map(call, ranges))
        if any(b < 0 for b in bad):
            raise N.NativeError("pve_expand_obs_host failed with %d" % min(bad))
        if sum(bad):
            raise ValueError("the factored observation holds %d invalid row codes" % sum(bad))
        return out[:n]

    def records(self, n=None):
        """Host buffers only: the agent records as a numpy structured array (``_native.RECORD_DTYPE``: reward, uid,
        lane, j, status, cpv, jerk_sum), a view of the pinned memory."""
        n = self._n if n is None else n
        return self.packed.numpy().view(N.RECORD_DTYPE).reshape(-1)[:n]

    @property
    def n_agents(self):
        """Total rows of this tick (synchronises)."""
        if self._n is None:
            self._n = int(self.agent_offset[-1].item())
        return self._n

    @property
    def actions(self):
        """``actions`` of the reference tuple: every row's own acceleration (TIS:290)."""
        return self.obs[:, :, 2]

    @property
    def done(self):
        return (self.status & N.ST_DONE) != 0


_POOLS = {}


def _pool(threads):
    if threads not in _POOLS:
        _POOLS[threads] = ThreadPoolExecutor(max_workers=threads, thread_name_prefix="pve_expand")
    return _POOLS[threads]


class BatchedScene:
    """B independent intersections resident on one GPU: the 12-lane one, or with ``SceneConfig(lane_num=4 / 8)`` the
    4- or 8-lane one.  ``neighbour_sources``: the step also writes ``StepOutputs.nbr_src`` (every geometry), which lets
    ``NStepFolder.push`` evaluate its target actor once per distinct row."""

    def __init__(self, n_envs, config=None, veh_cap=128, agent_cap=96, out_cap=None, device="cuda:0",
                 threads=0, _library=None, neighbour_sources=False, factored_obs=False, full_obs=True):
        self.cfg = config or SceneConfig()
        self.B, self.veh_cap, self.agent_cap = int(n_envs), int(veh_cap), int(agent_cap)
        self.out_cap = int(out_cap) if out_cap is not None else self.B * self.agent_cap
        self.device = torch.device(device)
        self.lib = N.load_library(_library)
        backend = self.lib.pve_backend().decode()
        if _library is None and backend != N.CUDA_BACKEND:
            raise N.NativeError("libpve_mcc.so reports backend %r, expected %r" % (backend, N.CUDA_BACKEND))
        if backend == N.CUDA_BACKEND:
            if self.device.type != "cuda":
                raise N.NativeError("the CUDA library needs a cuda device, got %s (there is no CPU fallback)" % device)
            if not torch.cuda.is_available():
                raise N.NativeError("no CUDA device is visible; the environment step has no CPU fallback")
        elif self.device.type != "cpu":
            raise N.NativeError("the test-only emulation library runs on host memory only")
        self.backend = backend
        self._h = C.c_void_p()
        ncfg = self.cfg.to_native(self.B, self.veh_cap, self.agent_cap, self.out_cap, threads)
        dev_index = self.device.index or 0
        rc = self.lib.pve_create(C.byref(ncfg), dev_index, C.byref(self._h))
        self._check(rc)
        # capacities are rounded up to a compiled capacity class; the class value is the array stride
        self.veh_cap = int(self.lib.pve_veh_cap(self._h))
        self.agent_cap = int(self.lib.pve_agent_cap(self._h))
        # factored_obs: the step also writes the factored observation (StepOutputs.row0_out / prev_row0 / obs_src;
        # 12-lane intersections only); full_obs=False: it does not write the 784-byte observation of every agent
        if factored_obs and self.cfg.lane_num != NLANE:
            raise ValueError("factored_obs exists for the 12-lane intersection only (lane_num=%d)" % self.cfg.lane_num)
        self.out = StepOutputs(self.B, self.out_cap, self.device, neighbour_sources=neighbour_sources,
                               factored=factored_obs, full_obs=full_obs, lib=self.lib)
        self._out_native = self.out.native()
        self._spawn = None
        self._counters = torch.zeros(16, dtype=torch.float64, device=self.device)

    # ---- plumbing ------------------------------------------------------------------------
    def _check(self, rc):
        if rc != 0:
            msg = self.lib.pve_last_error(self._h).decode() if self._h else "pve_create failed"
            raise N.NativeError("pve_mcc error %d: %s" % (rc, msg))

    def _stream(self):
        if self.device.type == "cuda":
            return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        return C.c_void_p(0)

    def close(self):
        if getattr(self, "_h", None):
            self.lib.pve_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def smem_bytes(self):
        return int(self.lib.pve_smem_bytes(self._h))

    @property
    def threads(self):
        return int(self.lib.pve_threads(self._h))

    @property
    def launch_info(self):
        """How a tick is launched (``pve_launch_info``): ``{"dual": bool, "small_veh_cap", "small_agent_cap",
        "small_threads", "small_smem_bytes"}``."""
        out = (C.c_int32 * 8)()
        self._check(self.lib.pve_launch_info(self._h, C.byref(out)))
        return {"dual": bool(out[0]), "small_veh_cap": out[1], "small_agent_cap": out[2], "small_threads": out[3],
                "small_smem_bytes": out[4]}

    # ---- reset: TrafficInteraction(arrive_time, ...) TIS:195-220 --------------------------
    def reset(self, arrive_time=None, warmup=True, spawn_ticks=None, intention_draws=None):
        """``arrive_time``: float64 seconds ``[K, 12]`` (shared) or ``[B, K, 12]`` (per intersection),
        the reference's ``arvTimeNewVeh`` table.  ``warmup`` advances each intersection to its first
        arrival like the reference constructor (TIS:214-220).

        ``lane_num=8`` only: ``intention_draws`` uint8 ``[K, 8]`` or ``[B, K, 8]``, entry ``[k][i]`` in {0, 1} = what the
        reference's ``random.randint(0, 1)`` returns for the k-th arrival of lane ``i`` (TIS:390; the reference seeds from
        OS entropy, so the draws are an input here).  Default: drawn with ``numpy.random.default_rng(0)``."""
        if spawn_ticks is None:
            arr = np.asarray(arrive_time, dtype=np.float64)
            if arr.ndim == 2:
                arr = arr[None]
            ticks = to_spawn_ticks(arr, self.cfg.deltaT)
            if ticks.shape[0] == 1 and self.B > 1:
                ticks = np.broadcast_to(ticks, (self.B,) + ticks.shape[1:])
        else:
            ticks = np.asarray(spawn_ticks, dtype=np.int32)
        nl = self.cfg.lane_num
        if nl != NLANE:
            assert ticks.shape[2] == nl, "lane_num=%d takes arrival tables with %d columns, got %r" % (nl, nl, ticks.shape)
            never = np.full(ticks.shape[:2] + (NLANE - nl,), 2**31 - 1, dtype=np.int32)     # lanes nl..11 do not exist
            ticks = np.concatenate([ticks, never], axis=2)
        if nl == 8:
            if intention_draws is None:
                dr = np.random.default_rng(0).integers(0, 2, size=(self.B, ticks.shape[1], 8), dtype=np.uint8)
            else:
                dr = np.asarray(intention_draws, dtype=np.uint8)
                if dr.ndim == 2:
                    dr = np.broadcast_to(dr[None], (self.B,) + dr.shape)
            assert dr.shape[0] == self.B and dr.shape[1] >= ticks.shape[1] and dr.shape[2] == 8, dr.shape
            full = np.zeros((self.B, ticks.shape[1], NLANE), np.uint8)
            full[:, :, :8] = dr[:, :ticks.shape[1]]
            self._draws = torch.from_numpy(full).to(self.device)
            self._check(self.lib.pve_set_intention_draws(self._h, self._draws.data_ptr()))
        assert ticks.shape[0] == self.B and ticks.shape[2] == NLANE, ticks.shape
        assert ticks.shape[1] < 65536, "arrival tables are limited to 65535 rows per lane"
        self._spawn = torch.from_numpy(np.ascontiguousarray(ticks)).to(self.device)
        self._check(self.lib.pve_reset(self._h, self._spawn.data_ptr(), ticks.shape[1], int(bool(warmup)),
                                       self._stream()))

    def reset_poisson(self, rate_veh_per_hour, seed, min_headway=1.0, warmup=True, first_env=0):
        """A new episode whose arrivals the step kernels generate on the device (``pve_reset_poisson``): per lane a
        Poisson stream with headways ``max(min_headway, Exp(mean = 3600 / rate_veh_per_hour))`` -- the distribution of
        ``synthetic_arrivals`` -- drawn from Philox with ``seed`` and the global intersection index
        ``first_env + b``.  No spawn table is built or kept, so an episode of any length costs O(B) memory, and a new
        episode with fresh traffic is one call with another seed.  ``arrivals.poisson_arrivals`` returns the same
        traffic as arrays.  With ``lane_num=8`` the intention draws come from the same stream.  A later ``reset`` with
        a table goes back to table mode.

        ``rate_veh_per_hour`` is one rate for every lane, or an array-like of rates broadcastable to ``[B, lane_num]``
        (``[B]``: one per intersection, ``[lane_num]``: one per lane, ``[B, lane_num]``) for ``pve_reset_poisson_rates``;
        equal rates give the same traffic either way.  A rank holding intersections ``[lo, hi)`` of a larger batch passes
        ``rates[lo:hi]`` with ``first_env=lo``."""
        rates = None
        if np.ndim(rate_veh_per_hour) == 0:
            rate = float(rate_veh_per_hour)
            if not (np.isfinite(rate) and rate > 0):
                raise ValueError("rate_veh_per_hour must be finite and > 0, got %r" % rate_veh_per_hour)
        else:
            rates = lane_rates(rate_veh_per_hour, self.B, self.cfg.lane_num)
            rate = 0.0                          # pve_reset_poisson_rates does not read it
        min_headway, seed, first_env = float(min_headway), int(seed), int(first_env)
        if not (np.isfinite(min_headway) and min_headway > 0):
            raise ValueError("min_headway must be finite and > 0, got %r" % min_headway)
        if not 0 <= seed < 2**64:
            raise ValueError("seed must be in [0, 2**64), got %r" % seed)
        if first_env < 0 or first_env + self.B > 2**32:
            raise ValueError("first_env must be >= 0 with first_env + n_envs <= 2**32, got %r" % first_env)
        if self.cfg.deltaT != 0.1:
            raise ValueError("Poisson arrivals use the reference's 0.1 s clock (deltaT=%r)" % self.cfg.deltaT)
        p = N.PvePoisson(seed, rate, min_headway, first_env)
        if rates is None:
            self._check(self.lib.pve_reset_poisson(self._h, C.byref(p), int(bool(warmup)), self._stream()))
        else:
            self._check(self.lib.pve_reset_poisson_rates(self._h, C.byref(p), rates.ctypes.data, int(bool(warmup)),
                                                         self._stream()))
        self._spawn = None           # the handle no longer reads the table

    # ---- step x V + scene_update + delete_vehicle ------------------------------------------
    def step(self, actions):
        """``actions``: float32 ``[B, veh_cap]`` on the scene's device; slot order is (lane, j), the
        order MAIN:398-406 iterates ``env.veh_info``.  Returns the reused ``StepOutputs``."""
        assert actions.dtype == torch.float32 and actions.is_contiguous()
        assert actions.shape == (self.B, self.veh_cap) and actions.device == self.device
        self.out._n = None
        self._check(self.lib.pve_step(self._h, actions.data_ptr(), C.byref(self._out_native), self._stream()))
        return self.out

    def make_host_outputs(self, pinned=True):
        """Pinned host mirrors of the output arrays for ``step_host``."""
        host = StepOutputs(self.B, self.out_cap, "cpu", lib=self.lib)
        if pinned and self.device.type == "cuda":
            host.pin()
        return host

    def step_host(self, actions_host, host_out, copy_obs=False):
        """One tick through HOST buffers (the end-to-end path): ``actions_host`` is a (pinned) CPU
        float32 ``[B, veh_cap]`` tensor; results land in ``host_out`` (from ``make_host_outputs``).
        Returns the number of agent rows of this tick.  With pinned buffers (the default of
        ``make_host_outputs``) the kernel works on them in place; the small arrays of ``self.out`` (reward, ids,
        cpv, status, jerk_sum, offsets, per-intersection counters) are then not refreshed, ``self.out.obs`` is."""
        assert actions_host.dtype == torch.float32 and actions_host.is_contiguous()
        assert actions_host.shape == (self.B, self.veh_cap) and actions_host.device.type == "cpu"
        n = int(self.lib.pve_next_agent_total(self._h, self._stream()))
        hn = host_out.native()
        self.out._n = None
        self._check(self.lib.pve_step_host(self._h, actions_host.data_ptr(), C.byref(self._out_native),
                                           C.byref(hn), 1 | (2 if copy_obs else 0), self._stream()))
        host_out._n = n
        self.out._n = n
        return n

    def make_async_buffers(self, factored=False, full_obs=None):
        """Three (device, pinned host) output pairs for ``step_host_async``: consecutive ticks take them in turn.
        ``factored``: with the factored observation (``copy_factored``); the device buffers then hold no ``obs`` unless
        ``full_obs`` is set, so the step does not write the 784-byte block of every agent."""
        full_obs = (not factored) if full_obs is None else bool(full_obs)
        pairs = []
        for _ in range(3):
            kw = dict(records_only=True, factored=factored, full_obs=full_obs, lib=self.lib)
            dev = StepOutputs(self.B, self.out_cap, self.device, **kw)
            host = StepOutputs(self.B, self.out_cap, "cpu", **kw).pin()
            pairs.append((dev, host, dev.native(), host.native()))      # the ctypes views are built once
        return pairs

    def step_host_async(self, actions_host, pair, copy_obs=False, copy_factored=False):
        """Enqueue one tick through host buffers without waiting (``pve_step_host_async``): actions by DMA from the
        pinned ``actions_host``, agent records / offsets / per-intersection counters (and the observations with
        ``copy_obs``, the factored observation with ``copy_factored``: 240 instead of 784 bytes per agent, rebuilt with
        ``host.expand_obs()``) by DMA into ``pair[1]`` while later ticks already run.  At most three ticks may be in
        flight; ``host_wait()`` returns the row count of the oldest one once its host buffers are complete."""
        assert actions_host.dtype == torch.float32 and actions_host.is_contiguous() and actions_host.is_pinned()
        assert actions_host.shape == (self.B, self.veh_cap)
        dev, host, dev_native, host_native = pair
        self._check(self.lib.pve_step_host_async(self._h, actions_host.data_ptr(), C.byref(dev_native),
                                                 C.byref(host_native), (2 if copy_obs else 0) | (4 if copy_factored else 0),
                                                 self._stream()))
        self._async_q = getattr(self, "_async_q", []) + [host]

    def host_wait(self):
        n = int(self.lib.pve_host_wait(self._h))
        if n < 0:
            self._check(n)
        host = self._async_q.pop(0)
        host._n = n
        return n, host

    def next_agent_total(self):
        return int(self.lib.pve_next_agent_total(self._h, self._stream()))

    # ---- state access (teacher forcing, snapshots; replaces reaching into env.veh_info) ------
    def _alloc_packed(self):
        B, cap = self.B, self.veh_cap
        return {"hdr": np.zeros(B, N.HDR_DTYPE), "meta": np.zeros((B, cap), N.META_DTYPE),
                "p": np.zeros((B, cap)), "v": np.zeros((B, cap)), "a": np.zeros((B, cap)),
                "jerk_sum": np.zeros((B, cap)), "row0": np.zeros((B, cap, OBS_W), np.float32)}

    def _view(self, packed):
        v = N.PveStateView()
        for k in ("hdr", "p", "v", "a", "jerk_sum", "meta", "row0"):
            assert packed[k].flags["C_CONTIGUOUS"]
            setattr(v, k, packed[k].ctypes.data)
        return v

    def get_state(self):
        packed = self._alloc_packed()
        self._check(self.lib.pve_get_state(self._h, C.byref(self._view(packed)), self._stream()))
        return N.unpack_state(packed, self.B, self.veh_cap)

    def set_state(self, st):
        n_ctrl = ((st["flags"] & N.F_CONTROL) != 0).sum(axis=1)
        if int(st["lane_n"].sum(axis=1).max()) > self.veh_cap - 1 or int(n_ctrl.max()) > self.agent_cap:
            raise ValueError("state does not fit veh_cap-1=%d vehicles / agent_cap=%d agents" % (self.veh_cap - 1, self.agent_cap))
        packed = N.pack_state(st, self.B, self.veh_cap)
        self._check(self.lib.pve_set_state(self._h, C.byref(self._view(packed)), self._stream()))
        if self.device.type == "cuda":
            torch.cuda.current_stream(self.device).synchronize()     # host arrays may go away

    # ---- device views for a device-side actor ---------------------------------------------
    def _wrap(self, ptr, shape, dtype, typestr):
        if self.device.type == "cuda":
            holder = type("DevArray", (), {})()
            holder.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False),
                                               "version": 2}
            return torch.as_tensor(holder, device=self.device)
        n = int(np.prod(shape))
        buf = (C.c_byte * (n * np.dtype(typestr).itemsize)).from_address(ptr)
        return torch.from_numpy(np.frombuffer(buf, dtype=np.dtype(typestr)).reshape(shape))

    def row0(self):
        """Stored observation row 0 of every vehicle slot, ``[B, veh_cap, 28]`` float32: the actor's
        input for the next tick (``veh["state"][0]``, MAIN:234-240).  Valid until the next ``step``."""
        return self._wrap(self.lib.pve_row0_dev(self._h), (self.B, self.veh_cap, OBS_W), torch.float32, "<f4")

    def row0_prev(self):
        """The rows the last ``step`` read, ``[B, veh_cap, 28]`` float32 in the slot order of that step's start: what
        a ``0x4000 | k`` code of ``StepOutputs.nbr_src`` names.  12 lanes: after every step; ``lane_num`` 4 / 8: after a
        step with ``neighbour_sources``.  Valid until the next ``step``, ``reset`` or ``set_state``."""
        return self._wrap(self.lib.pve_row0_prev_dev(self._h), (self.B, self.veh_cap, OBS_W), torch.float32, "<f4")

    def control_mask(self):
        """``veh["control"]`` of every slot, bool ``[B, veh_cap]`` (slots past the live count are False)."""
        meta = self._wrap(self.lib.pve_meta_dev(self._h), (self.B, self.veh_cap, 2), torch.int32, "<i4")
        hdr = self._wrap(self.lib.pve_hdr_dev(self._h), (self.B, N.HDR_DTYPE.itemsize // 4), torch.int32, "<i4")
        n_veh = hdr[:, 6]
        live = torch.arange(self.veh_cap, device=self.device)[None, :] < n_veh[:, None]
        return (((meta[:, :, 1] >> 24) & N.F_CONTROL) != 0) & live

    # ---- measurement -------------------------------------------------------------------------
    def set_profiling(self, on=True):
        self._check(self.lib.pve_set_profiling(self._h, int(bool(on))))

    def kernel_ms(self):
        """(step kernel ms, offset-scan kernel ms) of the last ``step``; waits for it to finish."""
        a, b = C.c_float(), C.c_float()
        self._check(self.lib.pve_kernel_ms(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    # ---- end-of-rollout statistics ----------------------------------------------------------
    def stats_tensor(self):
        """16 float64 counters on the device (see ``pve_counters``); all-reduce them across ranks."""
        self._check(self.lib.pve_stats(self._h, self._counters.data_ptr(), self._stream()))
        return self._counters

    ENV_STAT_NAMES = ("agent_steps", "vehicle_steps", "collided_agent_steps", "lock_events", "passed_jerk_sum", "reward_sum",
                      "reward_sq_sum", "removed", "env_steps", "q5_undefined")

    def env_stats(self):
        """The statistics per intersection (``pve_env_stats_dev``): float64 ``[B, 10]`` device view in the order of
        ``ENV_STAT_NAMES``; accumulated by the step kernel, so an evaluation loop needs no per-tick tallies."""
        return self._wrap(self.lib.pve_env_stats_dev(self._h), (self.B, len(self.ENV_STAT_NAMES)), torch.float64, "<f8")

    def stats(self):
        t = self.stats_tensor().cpu().numpy()
        return dict(zip(N.COUNTER_NAMES, t.tolist()))
