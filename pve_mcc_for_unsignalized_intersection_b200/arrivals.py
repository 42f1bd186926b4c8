"""Arrival-time tables: synthetic generator and conversion to integer spawn ticks.

The reference reads ``arvTimeNewVeh`` (float64 ``[K, 12]``, per-lane ascending arrival times in
seconds, zero-padded tail) from MATLAB files (main.py:228-229, 388-389) and spawns a vehicle on
lane ``i`` when ``current_time >= arrive_time[veh_rec[i]][i]`` (traffic_interaction_scene.py:379),
where ``current_time`` is a float64 that accumulates ``+= 0.1`` once per ``scene_update``
(traffic_interaction_scene.py:223).

On the device the comparison is done on integers: ``spawn_tick[k, i]`` is the first tick ``n``
whose accumulated clock satisfies the reference's comparison, so spawn indexing is bit-exact by
construction (SURVEY.md Q8).  Example: an arrival at 1.0 s spawns at tick 11, because ten
accumulated additions of 0.1 give 0.9999999999999999.
"""
import numpy as np

NLANE = 12
NEVER = np.int32(2**31 - 1)
MAX_TICK = 4_000_000          # arrivals later than this many ticks (111 h) are treated as NEVER


def reference_clock(n_ticks, delta_t=0.1):
    """``clock[n]`` = the reference's ``current_time`` after ``n`` scene updates (TIS:223)."""
    clock = np.zeros(n_ticks + 1, dtype=np.float64)
    # ufunc.accumulate is a strictly sequential left fold, i.e. the same additions in the same
    # order as ``t += delta_t`` (checked against a Python loop in tests/test_host_logic.py)
    np.add.accumulate(np.full(n_ticks, delta_t, dtype=np.float64), out=clock[1:])
    return clock


def to_spawn_ticks(arrive_time, delta_t=0.1, max_tick=None):
    """Convert arrival seconds ``[..., K, 12]`` to int32 spawn ticks of the same shape.

    The zero-padded tail of a lane -- its first entry that is not positive, or smaller than its predecessor -- and
    everything after it maps to ``NEVER``.  The reference would instead spawn one vehicle per tick from the padding and
    then raise ``IndexError`` at row ``K`` (SURVEY.md Q10); no shipped run reaches that point, and "table exhausted = no
    more arrivals" is the defined behaviour here.  Two EQUAL consecutive arrival times are valid arrivals: the reference
    spawns them on consecutive ticks (one vehicle per lane and tick, TIS:379), and so does the device.

    The last dimension is the number of lanes of the table: 12, or 8 / 4 for the 8- and 4-lane intersections (``lane_num``).
    """
    arr = np.asarray(arrive_time, dtype=np.float64)
    assert arr.shape[-1] in (NLANE, 8, 4), arr.shape
    K = arr.shape[-2]
    if max_tick is None:
        finite_max = float(arr.max()) if arr.size else 0.0
        max_tick = min(int(finite_max / delta_t) + 8, MAX_TICK)
    clock = reference_clock(max_tick, delta_t)
    # first n with clock[n] >= arr  (clock is strictly increasing)
    ticks = np.searchsorted(clock, arr, side="left").astype(np.int64)
    ticks = np.minimum(ticks, int(NEVER))
    ticks[ticks > max_tick] = int(NEVER)
    # padding: once a lane stops ascending, it never spawns again
    bad = arr <= 0
    if K > 1:
        bad[..., 1:, :] |= arr[..., 1:, :] < arr[..., :-1, :]
    bad = np.logical_or.accumulate(bad, axis=-2)
    ticks[bad] = int(NEVER)
    return ticks.astype(np.int32)


def synthetic_arrivals(n_envs, rate_veh_per_hour, horizon_s, seed=0, min_headway=1.0, rows=None):
    """Poisson-like arrival tables with the statistics of the shipped fixtures (SURVEY.md 8(d)).

    Per lane, independently: ``headway = max(min_headway, Exp(mean = 3600 / rate))``, first
    arrival drawn the same way, cumulative sum.  Returns float64 ``[n_envs, K, 12]`` whose rows
    cover at least ``horizon_s`` seconds on every lane.
    """
    mean = 3600.0 / float(rate_veh_per_hour)
    eff = min_headway + mean * np.exp(-min_headway / mean)      # E[max(h0, X)]
    if rows is None:
        rows = int(horizon_s / eff * 1.25) + 24
    rng = np.random.Generator(np.random.Philox(key=[seed, 0x5EED]))
    while True:
        head = rng.exponential(mean, size=(n_envs, rows, NLANE))
        np.maximum(head, min_headway, out=head)
        arr = np.cumsum(head, axis=1)
        if float(arr[:, -1, :].min()) > horizon_s:
            return arr
        rows = int(rows * 1.3) + 8


# ---- the Poisson arrival stream of BatchedScene.reset_poisson (csrc/arrivals.cuh), mirrored in numpy -------------------
_PHILOX_M0, _PHILOX_M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_PHILOX_W0, _PHILOX_W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
_U32 = np.uint64(0xFFFFFFFF)
# 2 / (2k + 1), k = 11 .. 1: the odd series of 2 atanh(s) (the same literals as csrc/arrivals.cuh)
_LOG_SERIES = (0.08695652173913043, 0.09523809523809523, 0.10526315789473684, 0.11764705882352941, 0.13333333333333333,
               0.15384615384615385, 0.18181818181818182, 0.2222222222222222, 0.2857142857142857, 0.4, 0.6666666666666666)
_LN2_HI, _LN2_LO = 6.93147180369123816490e-01, 1.90821492927058770002e-10
MAX_REC = 65535               # records from here on never spawn (veh_rec is 16 bits)


def philox4x32(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 on broadcastable arrays of 32-bit words (any integer dtype); returns four uint64 arrays of 32-bit
    words.  Counter 0, key 0 gives 6627e8d5 e169c58d bc57ac4c 9b00dbd8 (Random123's known-answer vector)."""
    c = [np.asarray(x).astype(np.uint64) & _U32 for x in (c0, c1, c2, c3)]
    k0, k1 = np.uint64(int(k0) & 0xFFFFFFFF), np.uint64(int(k1) & 0xFFFFFFFF)
    s32 = np.uint64(32)
    for _ in range(10):
        p0, p1 = _PHILOX_M0 * c[0], _PHILOX_M1 * c[2]
        c = [(p1 >> s32) ^ c[1] ^ k0, p1 & _U32, (p0 >> s32) ^ c[3] ^ k1, p0 & _U32]
        k0, k1 = (k0 + _PHILOX_W0) & _U32, (k1 + _PHILOX_W1) & _U32
    return c


def stream_log(u):
    """ln(u) for float64 u in [2^-53, 1] by the stream's own scheme (exact scaling to m in [sqrt(1/2), sqrt(2)),
    s = (m - 1) / (m + 1), odd series in s up to s^23, e * ln2 in two parts): + - * / only, so the device, the kernel
    emulation and numpy agree bit for bit.  Within 1 ulp of a correctly rounded log."""
    m, e = np.frexp(np.asarray(u, dtype=np.float64))
    low = m < 0.70710678118654752440
    m = np.where(low, m + m, m)
    dk = np.where(low, e - 1, e).astype(np.float64)
    f = m - 1.0
    s = f / (2.0 + f)
    z = s * s
    R = _LOG_SERIES[0]
    for c in _LOG_SERIES[1:]:
        R = c + z * R
    R = z * R
    hfsq = 0.5 * f * f
    return dk * _LN2_HI - ((hfsq - (s * (hfsq + R) + dk * _LN2_LO)) - f)


def poisson_arrivals(n_envs, rate_veh_per_hour, rows, seed, min_headway=1.0, first_env=0, lanes=NLANE):
    """The first ``rows`` records of every lane of the stream that ``BatchedScene.reset_poisson`` generates on the device,
    for global intersections ``first_env .. first_env + n_envs - 1``.  Returns ``(seconds, draws)``: float64 arrival
    times ``[n_envs, rows, lanes]`` and the lane_num = 8 intention draws (uint8 in {0, 1}) of the same records.
    ``rate_veh_per_hour`` is one rate for every lane (``reset_poisson(rate)``) or an array of rates read as
    ``lane_rates`` reads it (``reset_poisson(rates)``).

    Per record ``r`` of lane ``i`` of intersection ``e``: Philox4x32-10 with counter ``(e, i, r, 0)`` and key
    ``(seed & 0xffffffff, seed >> 32)`` gives ``w0..w3``; ``u = (((w0 << 21) | (w1 >> 11)) + 1) * 2**-53``; the headway is
    ``max(min_headway, -mean[b, i] * stream_log(u))`` with ``mean[b, i] = 3600 / rate[b, i]``; times are the running sums in record order;
    the draw is ``w2 & 1``.  ``to_spawn_ticks(seconds)`` gives the spawn ticks the device uses (which also never spawns
    a record past ``MAX_TICK`` or from record ``MAX_REC`` on).  The distribution is that of ``synthetic_arrivals``, the
    random stream is not."""
    seed = int(seed)
    e = (int(first_env) + np.arange(n_envs, dtype=np.uint64))[:, None, None]
    r = np.arange(rows, dtype=np.uint64)[None, :, None]
    i = np.arange(lanes, dtype=np.uint64)[None, None, :]
    w0, w1, w2, _ = philox4x32(e, i, r, np.uint64(0), seed & 0xFFFFFFFF, seed >> 32)
    x = (w0 << np.uint64(21)) | (w1 >> np.uint64(11))
    u = (x + np.uint64(1)).astype(np.float64) * 2.0 ** -53
    if np.ndim(rate_veh_per_hour) == 0:
        mean = 3600.0 / float(rate_veh_per_hour)
    else:
        mean = (3600.0 / lane_rates(rate_veh_per_hour, n_envs, lanes))[:, None, :]
    head = np.maximum(-mean * stream_log(u), float(min_headway))
    return np.add.accumulate(head, axis=1), (w2 & np.uint64(1)).astype(np.uint8)


def lane_rates(rates, n_envs, lanes):
    """Per-lane rates as ``reset_poisson`` and ``poisson_arrivals`` read them: ``[n_envs]`` (one per intersection),
    ``[lanes]`` (one per lane) or anything else that broadcasts to ``[n_envs, lanes]``.  Returns a C-contiguous float64
    ``[n_envs, lanes]`` array; raises ``ValueError`` for another shape, for a 1-D array when ``n_envs == lanes`` (one per
    intersection or one per lane?) and for an entry that is not finite and > 0, naming its intersection and lane."""
    a = np.asarray(rates, dtype=np.float64)
    if a.ndim == 1 and a.shape[0] == n_envs:
        if n_envs == lanes:
            raise ValueError("%d rates could be one per intersection or one per lane (n_envs == lane_num == %d): pass "
                             "them as [%d, 1] or [1, %d]" % (lanes, lanes, lanes, lanes))
        a = a[:, None]                          # one rate per intersection
    try:
        a = np.ascontiguousarray(np.broadcast_to(a, (n_envs, lanes)))
    except ValueError:
        raise ValueError("rates of shape %s do not broadcast to [n_envs, lane_num] = [%d, %d]"
                         % (np.shape(rates), n_envs, lanes)) from None
    bad = ~(np.isfinite(a) & (a > 0))
    if bad.any():
        b, i = np.argwhere(bad)[0]
        raise ValueError("every rate must be finite and > 0; intersection %d, lane %d has %r" % (b, i, a[b, i]))
    return a


def stress_arrivals(n_envs, horizon_s, headway=1.0):
    """Worst-case occupancy: every lane receives a vehicle every ``headway`` seconds."""
    rows = int(horizon_s / headway) + 4
    col = headway * np.arange(1, rows + 1, dtype=np.float64)
    return np.broadcast_to(col[None, :, None], (n_envs, rows, NLANE)).copy()
