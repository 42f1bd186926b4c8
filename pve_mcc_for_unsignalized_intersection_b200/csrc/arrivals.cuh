/*
 * arrivals.cuh -- the Poisson arrival stream that pve_reset_poisson generates on the device (include/pve_mcc.h).
 *
 * For global intersection e = first_env + b, lane i and arrival record r = 0, 1, ...:
 *   w0..w3 = Philox4x32-10(counter (e, i, r, 0), key (seed & 0xffffffff, seed >> 32))
 *   u      = (((w0 << 21) | (w1 >> 11)) + 1) * 2^-53                      in (0, 1]
 *   h_r    = max(min_headway, -mean[b][i] * pve_log_u(u)),  mean[b][i] = 3600 / rate[b][i] (float64, on the host)
 *   T_r    = T_{r-1} + h_r (float64, record order, T_{-1} = 0)
 *   spawn tick = the first n with clock[n] >= T_r (clock = the reference's accumulated 0.1 s clock, arrivals.py
 *                reference_clock); PVE_NEVER past PVE_MAX_TICK and from record PVE_MAX_REC on (veh_rec is 16 bits)
 *   lane_num = 8: the intention draw of record r is w2 & 1.
 * arrivals.poisson_arrivals is the independent numpy mirror of the same definition.  Only + - * / and exact scaling
 * enter pve_log_u (no libm / CUDA log, which differ in the last bits); with -fmad=false (device) and
 * -ffp-contract=off (emulation) the device, the emulation and numpy round identically.
 *
 * Included by scene_step.cuh after the PVE_HD / PVE_DEV macros.
 */
#pragma once

#define PVE_MAX_TICK 4000000     /* arrivals.MAX_TICK: later arrivals never spawn */
#define PVE_MAX_REC 65535        /* records from here on never spawn: veh_rec is 16 bits */

/* The generator's parameters: the kernel argument of the Poisson instantiations, in place of the spawn table. */
struct PvePoisson {
    const double *clock;      /* [PVE_MAX_TICK + 1] the reference's accumulated clock, built by the library */
    double *pend;             /* [B][12] arrival time T of record veh_rec[i] of lane i (the one next_spawn[i] is for) */
    double *mean;             /* [B][12] 3600 / rate of lane i of intersection b (pve_reset_poisson_rates) */
    double uniform_mean;      /* > 0: pve_reset_poisson's 3600 / rate, which the reset writes to every lane of `mean`;
                                 0: `mean` holds per-lane values already */
    double min_headway;       /* pve_poisson.min_headway */
    double clock_last;        /* clock[PVE_MAX_TICK] */
    uint32_t key0, key1;      /* seed & 0xffffffff, seed >> 32 */
    uint32_t first_env;       /* e = first_env + b */
    int32_t nlane;            /* lanes that exist: 12, or 4 / 8 (lanes past it never spawn) */
};

/* the kernel argument that carries the arrivals: the borrowed spawn table, or the generator */
template <bool POI> struct PveArrivalsT { typedef const int32_t *PVE_RESTRICT type; };
template <> struct PveArrivalsT<true> { typedef PvePoisson type; };

/* Philox4x32-10 (Salmon et al., SC'11; Random123): counter (c0, c1, c2, c3), key (k0, k1) -> w[4] */
PVE_HD void pve_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t w[4]) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
#ifdef __CUDA_ARCH__
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
#else
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0, hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
#endif
        c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    w[0] = c0; w[1] = c1; w[2] = c2; w[3] = c3;
}

/* ln(u) for u in [2^-53, 1]: u = 2^e * m with m in [sqrt(1/2), sqrt(2)) by exact scaling, f = m - 1,
 * s = f / (2 + f), ln(m) = f - f^2/2 + s (f^2/2 + R) with R = sum_{k=1..11} 2 s^2k / (2k + 1) (the odd series of
 * 2 atanh(s) up to s^23), plus e ln2 split into hi and lo parts (fdlibm's association order).  Within 1 ulp of a
 * correctly rounded log on (0, 1] (tests/test_poisson_arrivals.py); identical bits wherever it is compiled without
 * contraction. */
PVE_HD double pve_log_u(double u) {
#ifdef __CUDA_ARCH__
    const uint64_t bits = (uint64_t)__double_as_longlong(u);
#else
    uint64_t bits;
    memcpy(&bits, &u, sizeof bits);
#endif
    int e = (int)((bits >> 52) & 0x7FF) - 1022;                 /* u = 2^e * m, m in [0.5, 1): frexp */
    const uint64_t mb = (bits & 0x000FFFFFFFFFFFFFull) | 0x3FE0000000000000ull;
#ifdef __CUDA_ARCH__
    double m = __longlong_as_double((long long)mb);
#else
    double m;
    memcpy(&m, &mb, sizeof m);
#endif
    if (m < 0.70710678118654752440) { m = m + m; e -= 1; }
    const double dk = (double)e;
    const double f = m - 1.0;
    const double s = f / (2.0 + f), z = s * s;
    double R = 0.08695652173913043;                              /* 2/23 */
    R = 0.09523809523809523 + z * R;                             /* 2/21 */
    R = 0.10526315789473684 + z * R;                             /* 2/19 */
    R = 0.11764705882352941 + z * R;                             /* 2/17 */
    R = 0.13333333333333333 + z * R;                             /* 2/15 */
    R = 0.15384615384615385 + z * R;                             /* 2/13 */
    R = 0.18181818181818182 + z * R;                             /* 2/11 */
    R = 0.2222222222222222 + z * R;                              /* 2/9 */
    R = 0.2857142857142857 + z * R;                              /* 2/7 */
    R = 0.4 + z * R;                                             /* 2/5 */
    R = 0.6666666666666666 + z * R;                              /* 2/3 */
    R = z * R;
    const double hfsq = 0.5 * f * f;
    return dk * 6.93147180369123816490e-01 - ((hfsq - (s * (hfsq + R) + dk * 1.90821492927058770002e-10)) - f);
}

/* the Philox block of record r of lane i of intersection b */
PVE_HD void pve_arrival_block(const PvePoisson &A, int b, int i, int r, uint32_t w[4]) {
    pve_philox(A.first_env + (uint32_t)b, (uint32_t)i, (uint32_t)r, 0u, A.key0, A.key1, w);
}

/* the headway h_r of a block of a lane whose mean headway is `mean` (A.mean[b][i]) */
PVE_HD double pve_headway(const PvePoisson &A, double mean, const uint32_t w[4]) {
    const uint64_t x = ((uint64_t)w[0] << 21) | (uint64_t)(w[1] >> 11);
    const double u = (double)(x + 1) * 1.1102230246251565e-16;          /* 2^-53 */
    const double h = -mean * pve_log_u(u);
    return h > A.min_headway ? h : A.min_headway;
}

/* spawn tick of an arrival at T seconds: the first n with clock[n] >= T.  Up to PVE_MAX_TICK the accumulated clock
 * stays within 2.2e-5 s of n * 0.1, so the answer is n0, n0 + 1 or n0 + 2 with n0 = (int)(T * 10): two independent
 * reads of the clock, no search. */
PVE_HD int pve_spawn_tick_of(const PvePoisson &A, double T) {
    if (!(T <= A.clock_last)) return PVE_NEVER;
    int n = (int)(T * 10.0);
    n = n < PVE_MAX_TICK - 1 ? n : PVE_MAX_TICK - 1;
#ifdef __CUDA_ARCH__
    const double c0 = __ldg(A.clock + n), c1 = __ldg(A.clock + n + 1);
#else
    const double c0 = A.clock[n], c1 = A.clock[n + 1];
#endif
    return c0 >= T ? n : (c1 >= T ? n + 1 : n + 2);
}

/* arrival time T_r of record r (r < PVE_MAX_REC), summed from record 0 in record order: what pve_reset_poisson and
 * pve_set_state store as the pending time */
PVE_HD double pve_arrival_time(const PvePoisson &A, int b, int i, int r) {
    const double mean = A.mean[(size_t)b * PVE_NLANE + i];
    double T = 0.0;
    uint32_t w[4];
    for (int q = 0; q <= r; ++q) {
        pve_arrival_block(A, b, i, q, w);
        T = T + pve_headway(A, mean, w);
    }
    return T;
}

/* record `rec` of lane i has just become the next arrival (a spawn, or a reset): *pend goes from T_{rec-1} to
 * T_rec = T_{rec-1} + h_rec; returns its spawn tick.  `mean` is A.mean[b][i], which the step kernels load before the
 * call so that the load overlaps the Philox rounds; *pend is read after them (overlapping the log), which keeps the
 * small 12-lane step kernel within its 64 registers */
PVE_HD int pve_next_arrival(const PvePoisson &A, int b, int i, int rec, double *pend, double mean) {
    if (rec >= PVE_MAX_REC) return PVE_NEVER;
    uint32_t w[4];
    pve_arrival_block(A, b, i, rec, w);
    const double h = pve_headway(A, mean, w);
    const double T = *pend + h;
    *pend = T;
    return pve_spawn_tick_of(A, T);
}

/* pve_reset_poisson(_rates): record 0 becomes lane i's next arrival; lanes past A.nlane never spawn.  A uniform
 * reset writes the lane's mean here, so it needs neither an allocation nor a launch of its own. */
PVE_HD int pve_reset_lane(const PvePoisson &A, int b, int i) {
    const size_t q = (size_t)b * PVE_NLANE + i;
    if (A.uniform_mean > 0) A.mean[q] = A.uniform_mean;
    A.pend[q] = 0.0;
    return i < A.nlane ? pve_next_arrival(A, b, i, 0, A.pend + q, A.mean[q]) : PVE_NEVER;
}

/* pve_set_state: the pending time of record `rec` summed again from record 0 (the same additions in the same order
 * as the spawns that led there, so it is exact) and its spawn tick */
PVE_HD int pve_recount_lane(const PvePoisson &A, int b, int i, int rec) {
    if (i >= A.nlane || rec >= PVE_MAX_REC) return PVE_NEVER;
    const double T = pve_arrival_time(A, b, i, rec);
    A.pend[(size_t)b * PVE_NLANE + i] = T;
    return pve_spawn_tick_of(A, T);
}
