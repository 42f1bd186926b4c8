/*
 * scene_step4.cuh -- one tick of one 4-lane or 8-lane intersection (lane_num = 4 / 8), executed by one WARP.
 *
 * lane_num = 8 (two lanes per approach, 16 routes; TIS:100-145, 537-660, 1061-1249) runs the same control flow -- the
 * reference's scene_update is one loop for every lane_num != 12 -- with its own tables (Pve4Params), its own get_p
 * (pve8_world_xy), no get_state rewrite, `-1` routes skipped (TIS:236-237) and the intention of a new vehicle taken from
 * a table of draws (the reference calls random.seed() and random.randint(0, 1), TIS:382, 390: an input here).
 *
 * Replaces, for lane_num = 4, the reference's step() x V (traffic_interaction_scene.py "TIS" 1501-1539),
 * scene_update() (TIS:222-376) with get_virtual_distance (TIS:453-531), get_p (TIS:896-1062), get_state incl. its
 * rewrite of the virtual lane (TIS:1292-1338), virtual_lane_search_closer (TIS:1340-1405), check_lock
 * (TIS:1469-1499), add_new_veh (TIS:378-433) and delete_vehicle() (TIS:435-444).  SURVEY.md section 8(f), row N3.
 *
 * Why this is not the 12-lane kernel with other tables: a physical lane carries three routes (lane != route), the
 * virtual lane of a route also holds same-lane vehicles of the other routes (TIS:250-258), agents are processed lane by
 * lane, route by route, then by j, and for the left-turn routes every agent REWRITES the list that the agents after it
 * read (TIS:286-287 with 1301-1319).  That chain is inherently sequential over the agents of a route, and an
 * intersection is small (~30 vehicles, lists of ~20 entries), so the mapping is: one warp per intersection, agents in
 * the reference's order, the lanes of the warp over list entries / vehicles inside each step (membership, rank-count
 * stable sort, rewrite, six-nearest ranking, row copies).  Q3-Q5 of SURVEY.md 3.3 hold by construction here because
 * the order is the reference's own.
 *
 * The body uses three macros so that tests/emul/ can compile THE SAME SOURCE with g++ as a sequential emulation:
 *   P4_PAR(t, n)   independent iterations t = 0..n-1 (device: lanes stride over them; host: a plain loop)
 *   P4_ONE         executed once per intersection (device: lane 0)
 *   P4_SYNC        __syncwarp() / nothing
 * Float64 state arithmetic follows the reference's operation order (nvcc -fmad=false), so p, v, a, jerk_sum stay
 * bit-identical to it.
 */
#pragma once
#include "scene_step.cuh"

#define PVE4_NL 4
#define PVE4_ND 12
#define PVE4_MAXNL 8           /* lane_num = 8 */
#define PVE4_MAXND 16
#define PVE4_LC 128            /* list capacity (entries of one virtual lane) == vehicle slots staged per intersection */

#ifdef __CUDACC__
#define P4_PAR(t, n) for (int t = (int)(threadIdx.x & 31); t < (n); t += 32)
#define P4_ONE if ((threadIdx.x & 31) == 0)
#define P4_SYNC __syncwarp()
#else
#define P4_PAR(t, n) for (int t = 0; t < (n); ++t)
#define P4_ONE
#define P4_SYNC
#endif

struct Pve4Params {
    double dt, dt2, vm, vM, am, aM, v0, thr, lane_in, remove_p, cw, abs_am, two_abs_am, aspan;
    double L[3];
    double T[4][7], C[4][7], C2[4][7]; /* get_virtual_distance: member iff p1 - T > 0; vd = (|p1 - T| + C) - C2 (T = C = 0: vd = p1);
                                        * first index: route % ntype */
    double rw_k, rw_a, rw_b;           /* get_state rewrite (lane_num = 4): (alpha' - alpha) 3 cw, alpha' 3 cw, alpha 3 cw (TIS:1304-1316) */
    int8_t dir[PVE4_MAXNL][3];         /* direction[lane][intention], TIS:73-78 / 136-145 (-1: no such route) */
    int8_t l2l_pos[PVE4_MAXND][PVE4_MAXND];  /* position of route r in lane2lane[route] (TIS:58-71 / 107-123) or -1 */
    int8_t l2l_1[PVE4_MAXND];          /* lane2lane[route][1]: the route whose entries get_state rewrites (lane_num = 4) */
    int8_t int8[PVE4_MAXNL][2];        /* lane_num = 8: intention[lane][draw], TIS:125-134 */
    int32_t ntype;                     /* 3 (lane_num = 4) or 4 (lane_num = 8) */
    int32_t am_mask;                   /* lanes of `i in [2, 5, 8, 11]`, TIS:1519 */
    int32_t B, VC, K, zero_unctl;
    int64_t out_cap;
};

/* shared memory of one intersection (one warp) */
template <int LC_>      /* list capacity == vehicle slots staged per intersection: 64 (16 KB of shared memory less per CTA) or 128 */
struct alignas(16) Pve4SmemT {
    static constexpr int LC = LC_;
    pve_env_header h;                              /* first: copied with 16-byte accesses */
    double p[LC_], v[LC_], a[LC_], jerk[LC_], js[LC_], virdis[LC_];
    double lpos[LC_], tpos[LC_];          /* the current route's list (sorted); candidate positions */
    float rew[LC_];                            /* reward of output row g (overrides included) */
    int32_t uid[LC_], coll[LC_];
    uint32_t step[LC_];
    int16_t hdr[LC_];                          /* vir_header as a vehicle slot, or -1 */
    uint16_t lslot[LC_], agent[LC_], newpos[LC_], outrow[LC_], rowveh[LC_];
    uint8_t lane_of[LC_], intent[LC_], ctl[LC_], ctl_step[LC_], fin[LC_], del[LC_], lock[LC_],
        done_row[LC_], fin_now[LC_], ltag[LC_], tmem[LC_], ttag[LC_];
    int8_t lock_a[LC_];
    int32_t misc[16];                              /* see P4M_* */
    int32_t spawn[PVE4_MAXNL], spawn_int[PVE4_MAXNL], spawn_uid[PVE4_MAXNL];
    int16_t nbr[8];
    int32_t lane_off[PVE4_MAXNL + 1];
};
typedef Pve4SmemT<PVE4_LC> Pve4Smem;
enum { P4M_NA = 0, P4M_N, P4M_IDX, P4M_GOUT, P4M_COLL, P4M_LOCK, P4M_NREM, P4M_PASSED, P4M_PSTEP, P4M_Q5U, P4M_COLLAG, P4M_NSPAWN,
       P4M_NCTRL, P4M_SURV };

/* TIS:896-1062 get_p for lane_num = 4 (yaw is never read) */
PVE_DEV void pve4_world_xy(const Pve4Params &P, double p, int i, int m, double *x, double *y) {
    const double cw = P.cw;
    double u, w;                 /* the two coordinates before the lane's orientation is applied */
    int kind;                    /* 0: (u, w) pattern of the approach / straight leg, 1: left arc / exit, 2: right arc / exit */
    if (m == 1) {
        /* TIS:917-920, 958-961, 999-1002, 1040-1043 */
        if (i == 0) { *x = -1 * p + 2 * cw; *y = -1 * cw; } else if (i == 1) { *x = p - 2 * cw; *y = 1 * cw; }
        else if (i == 2) { *x = cw; *y = -1 * p + 2 * cw; } else { *x = -1 * cw; *y = p - 2 * cw; }
        return;
    }
    const double Lm = P.L[m];
    if (p > Lm) {                /* before the junction, TIS:901-904 etc. */
        u = p - Lm + 2 * cw;
        if (i == 0) { *x = -1 * u; *y = -1 * cw; } else if (i == 1) { *x = 1 * u; *y = 1 * cw; }
        else if (i == 2) { *x = 1 * cw; *y = -1 * u; } else { *x = -1 * cw; *y = 1 * u; }
        return;
    }
    (void)kind;
    if (p > 0) {
        const double R = (m == 0) ? 3 * cw : cw;
        const double b = p / R;                                      /* TIS:906, 927 */
        double s, c;
#ifdef __CUDACC__
        sincos(b, &s, &c);
#else
        s = sin(b); c = cos(b);
#endif
        if (m == 0) { s = s * 3 * cw; c = c * 3 * cw; } else { s = s * cw; c = c * cw; }
        if (m == 0) {            /* TIS:905-911, 946-952, 987-993, 1028-1034 */
            if (i == 0) { *x = 1 * (c - 2 * cw); *y = 1 * (2 * cw - s); } else if (i == 1) { *x = -1 * (c - 2 * cw); *y = -1 * (2 * cw - s); }
            else if (i == 2) { *x = 1 * (s - 2 * cw); *y = -1 * (2 * cw - c); } else { *x = -1 * (s - 2 * cw); *y = 1 * (2 * cw - c); }
        } else {                 /* TIS:926-932, 967-973, 1008-1014, 1049-1055 */
            if (i == 0) { *x = -1 * (2 * cw - c); *y = -1 * (2 * cw - s); } else if (i == 1) { *x = 1 * (2 * cw - c); *y = 1 * (2 * cw - s); }
            else if (i == 2) { *x = 1 * (2 * cw - s); *y = -1 * (2 * cw - c); } else { *x = -1 * (2 * cw - s); *y = 1 * (2 * cw - c); }
        }
        return;
    }
    w = -1 * p + 2 * cw;         /* past the exit point */
    if (m == 0) {                /* TIS:912-915, 953-956, 994-997, 1035-1038 */
        if (i == 0) { *x = cw; *y = w; } else if (i == 1) { *x = -1 * cw; *y = -1 * w; }
        else if (i == 2) { *x = -1 * w; *y = cw; } else { *x = 1 * w; *y = -1 * cw; }
    } else {                     /* TIS:933-936, 974-977, 1015-1018, 1056-1059 */
        if (i == 0) { *x = -1 * cw; *y = -1 * w; } else if (i == 1) { *x = 1 * cw; *y = w; }
        else if (i == 2) { *x = w; *y = -1 * cw; } else { *x = -1 * w; *y = 1 * cw; }
    }
}

/* TIS:1061-1249 get_p for lane_num = 8 (yaw is never read): even lanes turn left (m = 0) or go straight (m = 1), odd
 * lanes go straight or turn right (m = 2); a = i / 2 is the approach */
PVE_DEV void pve8_world_xy(const Pve4Params &P, double p, int i, int m, double *x, double *y) {
    const double cw = P.cw, a4 = 4 * cw;
    const int a = i >> 1;
    double u = 0, w = 0;         /* the pair before the approach's orientation is applied */
    int kind = 0;                /* how (u, w) maps to (x, y) for the four approaches */
    if ((i & 1) == 0) {
        if (m == 1) { u = p - a4; w = 1 * cw; kind = 0; }                                          /* TIS:1082-1085 ... */
        else if (p > P.L[0]) { u = p - P.L[0] + a4; w = 1 * cw; kind = 1; }                        /* TIS:1066-1069 ... */
        else if (p > 0) {
            const double b = p / (5 * cw);                                                         /* TIS:1071 */
            double s, c;
#ifdef __CUDACC__
            sincos(b, &s, &c);
#else
            s = sin(b); c = cos(b);
#endif
            s = s * 5 * cw; c = c * 5 * cw;
            /* TIS:1072-1075, 1119-1122, 1166-1169, 1213-1216 */
            if (a == 0) { *x = -1 * (c - a4); *y = -1 * (a4 - s); } else if (a == 1) { *x = -1 * (s - a4); *y = 1 * (a4 - c); }
            else if (a == 2) { *x = 1 * (c - a4); *y = 1 * (a4 - s); } else { *x = 1 * (s - a4); *y = -1 * (a4 - c); }
            return;
        } else {                                                                                   /* TIS:1078-1079 ... */
            const double q = -1 * p + a4;
            if (a == 0) { *x = -1 * cw; *y = -1 * q; } else if (a == 1) { *x = 1 * q; *y = -1 * cw; }
            else if (a == 2) { *x = cw; *y = q; } else { *x = -1 * q; *y = 1 * cw; }
            return;
        }
        if (kind == 0) {
            if (a == 0) { *x = u; *y = w; } else if (a == 1) { *x = -1 * cw; *y = u; }
            else if (a == 2) { *x = -1 * p + a4; *y = -1 * cw; } else { *x = 1 * cw; *y = -1 * p + a4; }
        } else {
            if (a == 0) { *x = 1 * u; *y = w; } else if (a == 1) { *x = -1 * cw; *y = 1 * u; }
            else if (a == 2) { *x = -1 * u; *y = -1 * cw; } else { *x = 1 * cw; *y = -1 * u; }
        }
        return;
    }
    if (m == 1) {                                                                                  /* TIS:1088-1091 ... */
        if (a == 0) { *x = p - a4; *y = 3 * cw; } else if (a == 1) { *x = -3 * cw; *y = p - a4; }
        else if (a == 2) { *x = -1 * p + a4; *y = -3 * cw; } else { *x = 3 * cw; *y = -1 * p + a4; }
        return;
    }
    if (p > P.L[2]) {                                                                              /* TIS:1094-1097 ... */
        u = p - P.L[2] + a4;
        if (a == 0) { *x = 1 * u; *y = 3 * cw; } else if (a == 1) { *x = -3 * cw; *y = 1 * u; }
        else if (a == 2) { *x = -1 * u; *y = -3 * cw; } else { *x = 3 * cw; *y = -1 * u; }
        return;
    }
    if (p > 0) {
        const double b = p / cw;                                                                   /* TIS:1099 */
        double s, c;
#ifdef __CUDACC__
        sincos(b, &s, &c);
#else
        s = sin(b); c = cos(b);
#endif
        s = s * cw; c = c * cw;
        /* TIS:1100-1103, 1147-1150, 1194-1197, 1241-1244 */
        if (a == 0) { *x = 1 * (a4 - c); *y = 1 * (a4 - s); } else if (a == 1) { *x = -1 * (a4 - s); *y = 1 * (a4 - c); }
        else if (a == 2) { *x = -1 * (a4 - c); *y = -1 * (a4 - s); } else { *x = 1 * (a4 - s); *y = -1 * (a4 - c); }
        return;
    }
    w = -1 * p + a4;                                                                               /* TIS:1106-1107 ... */
    if (a == 0) { *x = 3 * cw; *y = w; } else if (a == 1) { *x = -1 * w; *y = 3 * cw; }
    else if (a == 2) { *x = -3 * cw; *y = -1 * w; } else { *x = w; *y = -3 * cw; }
}

/* SRC: 8 slots of the in-place compaction of column c of the stored rows (pve4_step_block): DOWN = the vehicles that
 * move down or stay, k = k0 .. k0 + 7; else the ones that move up, k = k0 .. k0 - 7.  The loads of the 8 slots are all
 * issued before their stores. */
template <bool DOWN, class SMEM>
PVE_DEV void pve4_move_rows(const SMEM &M, float *rows_new, const float *rows_cur, const int c, const int k0, const int V) {
    float val[8];
    bool mv[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        const int k = DOWN ? k0 + u : k0 - u;
        mv[u] = (DOWN ? k < V : k >= 0) && !M.del[k] && (DOWN ? M.newpos[k] <= k : M.newpos[k] > k);
        if (mv[u]) val[u] = M.done_row[k] ? rows_new[(size_t)k * PVE_OBS_W + c] : rows_cur[(size_t)M.newpos[k] * PVE_OBS_W + c];
    }
#pragma unroll
    for (int u = 0; u < 8; ++u)
        if (mv[u]) rows_new[(size_t)M.newpos[DOWN ? k0 + u : k0 - u] * PVE_OBS_W + c] = val[u];
}

/* one tick of intersection b.  The caller passes the stored rows of the tick's start as S.row0[0] and the other buffer as
 * S.row0[1].  rows_cur: the stored rows (indexed by the vehicle slots of the tick's start); rows_new: the rows computed
 * this tick (same indexing).
 *   SRC = false: rows_new is scratch; rows_cur is rewritten at the end for the next tick (slot order after removals).
 *   SRC = true:  also writes pve_outputs.nbr_src.  rows_cur is only read, so it still holds the rows this tick read when
 *                the tick ends (pve_nstep_push_scene needs them); rows_new is compacted in place into the stored rows of
 *                the next tick, and the caller swaps the two buffers.  Both leave the same rows in every slot below the
 *                new vehicle count. */
template <int NLN, bool POI, bool SRC, class SMEM>      /* lane_num: 4 or 8; POI: Poisson arrivals (see pve_step_block); SMEM: Pve4SmemT<64> or <128> */
PVE_DEV void pve4_step_block(const Pve4Params &P, const PveState &S, const pve_outputs &O,
                             const typename PveArrivalsT<POI>::type arr, const uint8_t *PVE_RESTRICT draws,
                             const float *PVE_RESTRICT actions, const int b, SMEM &M, const int64_t obase) {
    constexpr int PVE4_NLX = NLN;
    const size_t vbase = (size_t)b * (size_t)P.VC;
    float *const rows_cur = S.row0[0] + vbase * PVE_OBS_W;
    float *const rows_new = S.row0[1] + vbase * PVE_OBS_W;

    /* ---- load -------------------------------------------------------------------------------------------------- */
    P4_PAR(t, (int)(PVE_HDR_BYTES / 16)) ((pve_v4 *)&M.h)[t] = ((const pve_v4 *)(S.hdr + b))[t];
    P4_SYNC;
    P4_ONE {
        int o = 0;
        for (int i = 0; i < PVE4_NLX; ++i) { M.lane_off[i] = o; o += M.h.lane_n[i]; }
        M.lane_off[PVE4_NLX] = o;
        for (int q = 0; q < 16; ++q) M.misc[q] = 0;
    }
    P4_SYNC;
    const int V = M.lane_off[PVE4_NLX];
    P4_PAR(k, V) {
        M.p[k] = S.p[vbase + k]; M.v[k] = S.v[vbase + k]; M.a[k] = S.a[vbase + k]; M.js[k] = S.js[vbase + k];
        const pve_veh_meta mt = S.meta[vbase + k];
        const uint32_t fl = mt.packed >> 24;
        M.uid[k] = mt.uid;
        M.step[k] = mt.packed & 0xFFFFu;
        M.coll[k] = (int32_t)((mt.packed >> 16) & 0xFFu);
        M.ctl[k] = (fl & PVE_F_CONTROL) ? 1 : 0; M.fin[k] = (fl & PVE_F_FINISH) ? 1 : 0;
        M.lock[k] = (fl & PVE_F_LOCK) ? 1 : 0; M.lock_a[k] = (int8_t)((int)((fl >> 3) & 3u) - 1);
        M.intent[k] = (uint8_t)((fl >> 5) & 3u);
        int i = 0;
        for (int q = 1; q < PVE4_NLX; ++q) if (k >= M.lane_off[q]) i = q;
        M.lane_of[k] = (uint8_t)i;
        M.hdr[k] = -1; M.virdis[k] = 100.0; M.del[k] = 0; M.jerk[k] = 0.0; M.done_row[k] = 0; M.fin_now[k] = 0;
    }
    P4_SYNC;

    /* ---- step() for every vehicle: one lane of the warp per physical lane, its vehicles in order (the rear-end rule
     *      reads the already stepped leader, TIS:1509-1516) ---------------------------------------------------------- */
    P4_PAR(i, PVE4_NLX) {
        for (int k = M.lane_off[i]; k < M.lane_off[i + 1]; ++k) {
            const int j = k - M.lane_off[i];
            const double act = (P.zero_unctl && !M.ctl[k]) ? 0.0 : (double)actions[vbase + k];
            double ta = fmin(P.aM, fmax(P.am, act));                                              /* TIS:1502 */
            if (M.lock[k] && M.lock_a[k] != 0 && M.p[k] > 70.0) ta = M.a[k] + (double)M.lock_a[k]; /* TIS:1503-1505 */
            M.lock[k] = 0; M.lock_a[k] = 0;                                                       /* TIS:1506-1507 */
            if (j > 0 && M.v[k - 1] < M.v[k] && M.ctl[k - 1] && M.ctl[k]) {                       /* TIS:1509-1516 */
                const double v = M.v[k], vf = M.v[k - 1];
                const double d_safe = v * 0.4 + (v * v - vf * vf) / P.two_abs_am - (v - vf) * P.vm / P.abs_am;
                if (M.p[k] - M.p[k - 1] < d_safe) ta = P.am;
            }
            if (M.h.head_lane[i] == i && M.h.head_j[i] == j) ta = P.aM;                           /* TIS:1517: virtual_lane_4[i], the LANE index */
            if ((P.am_mask >> i) & 1) ta = P.aM;                                                  /* TIS:1519: `i in [2, 5, 8, 11]` */
            ta = fmin(P.aM, fmax(P.am, ta));                                                      /* TIS:1521 */
            M.jerk[k] = ta - M.a[k];
            M.a[k] = ta;
            M.p[k] = M.p[k] - M.v[k] * P.dt - 0.5 * M.a[k] * P.dt2;                               /* TIS:1528-1529 */
            M.v[k] = fmin(P.vM, fmax(M.v[k] + M.a[k] * P.dt, P.vm));                              /* TIS:1530-1531 */
            M.step[k] = M.step[k] < 0xFFFFu ? M.step[k] + 1 : M.step[k];                          /* TIS:1533 */
            if (!M.ctl[k]) M.v[k] = P.v0;                                                         /* TIS:1535 */
            M.ctl_step[k] = M.ctl[k];
        }
    }
    P4_SYNC;
    P4_ONE {      /* self.virtual_lane: the controlled vehicles in step order (TIS:1539) */
        int na = 0;
        for (int k = 0; k < V; ++k) if (M.ctl_step[k]) M.agent[na++] = (uint16_t)k;
        M.misc[P4M_NA] = na;
    }
    P4_SYNC;
    const int NA = M.misc[P4M_NA];
    const bool out_ok = obase + NA <= P.out_cap;

    /* ---- scene_update: lane by lane, route by route, vehicle by vehicle (TIS:233-361) ---------------------------------- */
    for (int i = 0; i < PVE4_NLX; ++i) {
        if (M.lane_off[i + 1] == M.lane_off[i]) continue;                                         /* TIS:234 */
        for (int m = 0; m < 3; ++m) {
            const int route = P.dir[i][m];
            if (route < 0) continue;                                                              /* TIS:236-237 (lane_num = 8) */
            /* membership and virtual position of every controlled vehicle (TIS:240-270) */
            P4_PAR(g, NA) {
                const int k = M.agent[g], l = M.lane_of[k], it = M.intent[k];
                const int r = P.dir[l][it];
                int mem = 0, tag = route;
                double pos = M.p[k];
                if (l == i) {
                    if (r == route) mem = 1;                                                      /* TIS:246-249 */
                    else if (M.p[k] - P.L[it] > 0) { pos = M.p[k] - P.L[it] + P.L[m]; mem = 1; }   /* TIS:252-258 */
                } else {
                    const int kk = P.l2l_pos[route][r];
                    if (kk >= 0) {                                                                /* TIS:259-270, 453-531 */
                        const int ty = route % P.ntype;
                        const double T = P.T[ty][kk], C = P.C[ty][kk];
                        const double delta = M.p[k] - T;
                        if (delta > 0) { mem = 1; tag = r; pos = (T == 0.0 && C == 0.0) ? M.p[k] : (fabs(delta) + C) - P.C2[ty][kk]; }
                    }
                }
                M.tmem[g] = (uint8_t)mem; M.ttag[g] = (uint8_t)tag; M.tpos[g] = pos;
            }
            P4_SYNC;
            /* stable sort by position (TIS:271): rank = members that precede in (pos, step order) */
            P4_PAR(g, NA) {
                if (M.tmem[g]) {
                    int rank = 0;
                    for (int q = 0; q < NA; ++q)
                        if (M.tmem[q] && (M.tpos[q] < M.tpos[g] || (M.tpos[q] == M.tpos[g] && q < g))) ++rank;
                    M.lpos[rank] = M.tpos[g]; M.lslot[rank] = M.agent[g]; M.ltag[rank] = M.ttag[g];
                }
            }
            P4_ONE {
                int n = 0;
                for (int q = 0; q < NA; ++q) n += M.tmem[q];
                M.misc[P4M_N] = n;
            }
            P4_SYNC;
            const int n = M.misc[P4M_N];
            P4_ONE {      /* virtual_lane_4[route][0], read by next tick's step() (the rewrite below keeps the list order) */
                if (route < PVE_NLANE) {      /* (lane_num = 8 has 16 routes; step() reads the heads of routes 0-7 only) */
                    if (n > 0) { const int kh = M.lslot[0]; M.h.head_lane[route] = (int8_t)M.lane_of[kh]; M.h.head_j[route] = (uint8_t)(kh - M.lane_off[M.lane_of[kh]]); }
                    else { M.h.head_lane[route] = -1; M.h.head_j[route] = 0; }
                }
            }
            /* the vehicles of this route, in lane order */
            for (int k = M.lane_off[i]; k < M.lane_off[i + 1]; ++k) {
                if (M.intent[k] != m) continue;                                                   /* TIS:275 */
                if (M.ctl[k]) {
                    /* ---- get_state (TIS:1292-1338) ---- */
                    P4_PAR(s, n) if (M.lslot[s] == k) M.misc[P4M_IDX] = s;
                    P4_SYNC;
                    const int idx = M.misc[P4M_IDX];
                    const double ego0 = M.lpos[idx];
                    if (NLN == 4 && route % 3 == 0) {                                             /* TIS:1301-1319: the rewrite, kept for later agents */
                        const int tag = P.l2l_1[route];
                        P4_PAR(s, n) {
                            if (M.ltag[s] == tag) {
                                const double ori_p = M.lpos[s] + P.rw_k;
                                double np_;
                                if (ego0 < ori_p) { np_ = ori_p - P.rw_a + P.rw_b; if (np_ < ego0) np_ = ego0 + 1; }
                                else { np_ = ori_p + P.rw_a - P.rw_b; if (np_ > ego0) np_ = ego0 - 1; }
                                M.lpos[s] = np_;
                            }
                        }
                        P4_SYNC;
                    }
                    const double pe = M.lpos[idx];
                    /* ---- virtual_lane_search_closer, "closer" (TIS:1340-1405) ---- */
                    P4_ONE {
                        if (idx == 0) { M.hdr[k] = -1; M.virdis[k] = 100.0; }
                        else { M.hdr[k] = (int16_t)M.lslot[idx - 1]; M.virdis[k] = M.lpos[idx] - M.lpos[idx - 1]; }
                        for (int q = 0; q < PVE_NNBR; ++q) M.nbr[q] = -1;
                    }
                    P4_SYNC;
                    P4_PAR(s, n) {
                        if (s != idx) {
                            const double d = fabs(M.lpos[s] - pe);
                            int rank = 0;
                            for (int q = 0; q < n; ++q) {
                                if (q == idx || q == s) continue;
                                const double dq = fabs(M.lpos[q] - pe);
                                if (dq < d || (dq == d && q < s)) ++rank;
                            }
                            if (rank < PVE_NNBR) M.nbr[rank] = (int16_t)s;
                        }
                    }
                    P4_SYNC;
                    /* ---- rows: row 0 from the list, rows 1..6 = the neighbours' stored rows (Q3) ---- */
                    const int g_out = M.misc[P4M_GOUT];
                    float *const orow = (out_ok && O.obs) ? O.obs + (size_t)(obase + g_out) * (PVE_OBS_H * PVE_OBS_W) : nullptr;
                    P4_PAR(q, PVE_OBS_H) {
                        float r0, r1, r2, r3;
                        if (q == 0) { r0 = (float)pe; r1 = (float)M.v[k]; r2 = (float)M.a[k]; r3 = (float)route; }        /* TIS:1336 */
                        else {
                            const int s = M.nbr[q - 1];
                            if (s >= 0) {
                                const int ks = M.lslot[s];
                                r0 = (float)M.lpos[s]; r1 = (float)M.v[ks]; r2 = (float)M.a[ks];                          /* TIS:1330 */
                                r3 = (float)P.dir[M.lane_of[ks]][M.intent[ks]];
                            } else { r0 = r1 = r2 = r3 = 0.f; }                                                           /* TIS:1334 */
                        }
                        float *dst = rows_new + (size_t)k * PVE_OBS_W + 4 * q;
                        dst[0] = r0; dst[1] = r1; dst[2] = r2; dst[3] = r3;
                        if (orow) { orow[4 * q] = r0; orow[4 * q + 1] = r1; orow[4 * q + 2] = r2; orow[4 * q + 3] = r3; }
                    }
                    if (orow) {
                        P4_PAR(x, PVE_NNBR * PVE_OBS_W) {
                            const int q = x / PVE_OBS_W, c = x - q * PVE_OBS_W;
                            const int s = M.nbr[q];
                            float val = 0.f;
                            if (s >= 0) {
                                const int ks = M.lslot[s];
                                val = (M.done_row[ks] ? rows_new : rows_cur)[(size_t)ks * PVE_OBS_W + c];                  /* TIS:1332 */
                            }
                            orow[(q + 1) * PVE_OBS_W + c] = val;
                        }
                    }
                    P4_SYNC;
                    /* ---- reward, collision, bookkeeping of the agent (TIS:293-340) ---- */
                    P4_ONE {
                        if constexpr (SRC) {      /* pve_outputs.nbr_src: the source of each row copied above */
                            if (out_ok && O.nbr_src) {
                                uint32_t w4[4];
                                w4[0] = (uint32_t)g_out;
                                for (int q = 1; q < 8; ++q) {
                                    const int s = q < PVE_OBS_H ? (int)M.nbr[q - 1] : -1;
                                    uint32_t v = 0xFFFFu;
                                    if (s >= 0) {
                                        const int ks = M.lslot[s];
                                        v = M.done_row[ks] ? (uint32_t)M.outrow[ks] : (0x4000u | (uint32_t)ks);
                                    }
                                    if (q & 1) w4[q >> 1] |= v << 16; else w4[q >> 1] = v;
                                }
                                pve_v4 nb; nb.x = w4[0]; nb.y = w4[1]; nb.z = w4[2]; nb.w = w4[3];
                                ((pve_v4 *)O.nbr_src)[obase + g_out] = nb;
                            }
                        }
                        M.done_row[k] = 1;
                        const int s0 = M.nbr[0];
                        const int k0 = s0 >= 0 ? (int)M.lslot[s0] : 0;
                        M.rew[g_out] = pve_reward(P.vm, P.aspan, M.p[k], M.v[k], M.jerk[k] / P.dt, s0 >= 0, s0 >= 0 ? M.lpos[s0] : 0.0,
                                                  s0 >= 0 ? M.v[k0] : 0.0);
                        M.js[k] += fabs(M.jerk[k] / P.dt);                                        /* TIS:321 */
                        if (s0 >= 0) {                                                            /* TIS:322-334 */
                            double x0, y0, x1, y1;
                            if (NLN == 4) {
                                pve4_world_xy(P, M.p[k], i, m, &x0, &y0);
                                pve4_world_xy(P, M.p[k0], M.lane_of[k0], M.intent[k0], &x1, &y1);
                            } else {
                                pve8_world_xy(P, M.p[k], i, m, &x0, &y0);
                                pve8_world_xy(P, M.p[k0], M.lane_of[k0], M.intent[k0], &x1, &y1);
                            }
                            const double dx = x1 - x0, dy = y1 - y0;
                            if (sqrt(dx * dx + dy * dy) < P.thr) { M.coll[k] += 1; M.coll[k0] += 1; }
                        }
                        if (M.fin[k]) M.ctl[k] = 0;                                               /* TIS:335-336 */
                        M.misc[P4M_COLL] += M.coll[k];                                            /* TIS:337 */
                        if (M.coll[k] > 0) M.misc[P4M_COLLAG] += 1;
                        if (out_ok && O.cpv) O.cpv[obase + g_out] = M.coll[k];                    /* TIS:339 */
                        M.outrow[k] = (uint16_t)g_out;
                        M.rowveh[g_out] = (uint16_t)k;
                        M.misc[P4M_GOUT] = g_out + 1;
                    }
                    P4_SYNC;
                }
                /* ---- flags of the vehicle, controlled or not (TIS:341-359) ---- */
                P4_ONE {
                    const int last = M.misc[P4M_GOUT] - 1;                                        /* reward[-1] */
                    if (M.p[k] < P.remove_p || M.coll[k] > 0) {
                        if (M.coll[k] > 0) { if (last >= 0) M.rew[last] = -10.f; else M.misc[P4M_Q5U] += 1; }   /* TIS:345-346 */
                        M.del[k] = 1; M.misc[P4M_NREM] += 1;                                      /* TIS:347-348 */
                        M.hdr[k] = -1;
                    } else if (M.p[k] < 0 && M.ctl[k]) {                                          /* TIS:350-359 */
                        M.fin[k] = 1; M.fin_now[k] = 1; M.ctl[k] = 0; M.hdr[k] = -1; M.lock[k] = 0;
                        M.misc[P4M_PASSED] += 1;
                        if (last >= 0) M.rew[last] = 5.f;
                        M.misc[P4M_PSTEP] += (int)M.step[k];
                    }
                }
                P4_SYNC;
            }
        }
    }

    /* ---- arrivals (TIS:378-433; after each lane's vehicles, i.e. in lane order; the newcomers take no part in this
     *      tick) and the survivors' new slots (delete_vehicle, TIS:435-444) ----------------------------------------- */
    P4_ONE {
        const int tick = M.h.tick + 1;                                                            /* TIS:223 */
        int surv = 0, nctrl = 0;
        for (int k = 0; k < V; ++k) if (!M.del[k]) { ++surv; nctrl += M.ctl[k]; }
        int granted = 0, pos = 0, k = 0;
        for (int i = 0; i < PVE4_NLX; ++i) {
            int cnt = 0;
            for (; k < M.lane_off[i + 1]; ++k) if (!M.del[k]) { M.newpos[k] = (uint16_t)pos++; ++cnt; }
            M.spawn[i] = 0;
            if (tick >= M.h.next_spawn[i] && cnt < 255) {                                         /* TIS:379 */
                if (surv + granted < P.VC && surv + granted < SMEM::LC) {
                    M.spawn[i] = 1 + pos;                         /* slot + 1 */
                    if (NLN == 4) {
                        M.spawn_int[i] = M.h.pad_[0] % 3;         /* TIS:387: intention_re % 3 */
                        M.h.pad_[0] = (uint8_t)((M.h.pad_[0] + 1) % 3);
                    } else if constexpr (POI) {                   /* TIS:390: the draw of the record is w2 & 1 of its block */
                        uint32_t w[4];
                        pve_arrival_block(arr, b, i, M.h.veh_rec[i], w);
                        M.spawn_int[i] = P.int8[i][w[2] & 1];
                    } else {                                      /* TIS:390: intention[i][random.randint(0, 1)], the draw is an input */
                        const int dr = draws ? (int)(draws[((size_t)b * P.K + M.h.veh_rec[i]) * PVE_NLANE + i] & 1) : 0;
                        M.spawn_int[i] = P.int8[i][dr];
                    }
                    M.spawn_uid[i] = M.h.id_seq + granted;        /* TIS:433 */
                    ++pos; ++cnt; ++granted;
                    const int rec = (int)M.h.veh_rec[i] + 1;      /* TIS:430 */
                    M.h.veh_rec[i] = (uint16_t)rec;
                    if constexpr (POI) {
                        const size_t q = (size_t)b * PVE_NLANE + i;
                        M.h.next_spawn[i] = pve_next_arrival(arr, b, i, rec, arr.pend + q, arr.mean[q]);
                    } else {
                        M.h.next_spawn[i] = (rec < P.K) ? arr[((size_t)b * P.K + rec) * PVE_NLANE + i] : PVE_NEVER;
                    }
                } else M.h.overflow += 1;
            }
            M.h.lane_n[i] = (uint8_t)cnt;
        }
        if (!out_ok) M.h.overflow += 1;
        M.h.tick = tick;
        M.h.id_seq += granted;
        M.h.passed_veh += M.misc[P4M_PASSED];
        M.h.passed_step_total += M.misc[P4M_PSTEP];
        M.h.n_veh = surv + granted;
        M.h.n_ctrl = nctrl + granted;
        M.misc[P4M_NSPAWN] = granted;
    }
    P4_SYNC;

    /* ---- deadlock scan (TIS:365-370 + 1469-1499): every controlled vehicle follows vir_header for up to 10 hops; the
     *      first member of a ring in (lane, j) order reports it ------------------------------------------------------- */
    P4_PAR(k, V) {
        if (M.ctl[k]) {
            int t = k, len = 0;
            for (int hop = 1; hop <= 10; ++hop) {                                                 /* TIS:1470-1478 */
                t = (t >= 0 && len == 0) ? (int)M.hdr[t] : -1;
                len = (t == k) ? hop : len;
            }
            if (len > 0) {
                M.lock[k] = 1;                                                                    /* TIS:1482 */
                int mn = k;
                t = k;
                for (int hop = 0; hop < len; ++hop) { t = M.hdr[t]; mn = t < mn ? t : mn; }
                if (mn == k) {
                    PVE_ATOMIC_ADD(&M.misc[P4M_LOCK], 1);
                    /* record_.sort() (TIS:1492): (vir_dis, follower) is the whole key; walk the ring once per position */
                    double last_d = -1.0e300, sum = 0, first_d = 0;
                    int last_o = -1, first_o = -1;
                    for (int x = 0; x < len; ++x) {
                        double best_d = 1.0e300;
                        int best_o = 0x7FFFFFFF;
                        t = k;
                        for (int hop = 0; hop < len; ++hop) {
                            const double dd = M.virdis[t];
                            const bool after = dd > last_d || (dd == last_d && t > last_o);
                            const bool better = dd < best_d || (dd == best_d && t < best_o);
                            if (after && better) { best_d = dd; best_o = t; }
                            t = M.hdr[t];
                        }
                        sum = sum + best_d;                                                       /* TIS:1495 sum(dis) */
                        if (x == 0) { first_d = best_d; first_o = best_o; }
                        last_d = best_d; last_o = best_o;
                    }
                    if (first_d < P.thr || sum / (double)len < P.thr + 3) {                       /* TIS:1495 */
                        M.lock_a[first_o] = 1;                                                    /* TIS:1496 */
                        M.lock_a[M.hdr[first_o]] = -1;                                            /* TIS:1497 */
                    }
                }
            }
        }
    }
    P4_SYNC;

    /* ---- outputs of the agents (final flags), state write-back, header, statistics ------------------------------------ */
    const int G = M.misc[P4M_GOUT];
    if (out_ok) {
        P4_PAR(g, G) {
            const int k = M.rowveh[g];
            const int64_t row = obase + g;
            if (O.reward) O.reward[row] = M.rew[g];
            if (O.ids) {
                pve_v4 id; id.x = (uint32_t)b; id.y = M.lane_of[k]; id.z = (uint32_t)(k - M.lane_off[M.lane_of[k]]); id.w = (uint32_t)M.uid[k];
                ((pve_v4 *)O.ids)[row] = id;
            }
            const uint8_t st = (uint8_t)((M.del[k] ? (PVE_ST_DONE | PVE_ST_REMOVED) : 0) | (M.fin_now[k] ? (PVE_ST_DONE | PVE_ST_FINISHED) : 0));
            if (O.status) O.status[row] = st;
            if (O.jerk_sum) O.jerk_sum[row] = (float)M.js[k];
            if (O.packed) {
                const uint32_t c8 = M.coll[k] > 255 ? 255u : (uint32_t)M.coll[k];
                pve_v4 rec;
                rec.x = pve_fbits(M.rew[g]); rec.y = (uint32_t)M.uid[k];
                rec.z = (uint32_t)M.lane_of[k] | ((uint32_t)(k - M.lane_off[M.lane_of[k]]) << 8) | ((uint32_t)st << 16) | (c8 << 24);
                rec.w = pve_fbits((float)M.js[k]);
                ((pve_v4 *)O.packed)[row] = rec;
            }
        }
    }
    P4_PAR(k, V) {
        if (!M.del[k]) {
            const size_t o = vbase + (size_t)M.newpos[k];
            S.p[o] = M.p[k]; S.v[o] = M.v[k]; S.a[o] = M.a[k]; S.js[o] = M.js[k];
            pve_veh_meta mt;
            mt.uid = M.uid[k];
            const uint32_t c8 = M.coll[k] > 255 ? 255u : (uint32_t)M.coll[k];
            const uint32_t fl = (M.ctl[k] ? PVE_F_CONTROL : 0) | (M.fin[k] ? PVE_F_FINISH : 0) | (M.lock[k] ? PVE_F_LOCK : 0)
                                | ((uint32_t)(M.lock_a[k] + 1) << 3) | ((uint32_t)M.intent[k] << 5);
            mt.packed = M.step[k] | (c8 << 16) | (fl << 24);
            S.meta[o] = mt;
            if (!SRC && M.done_row[k])
                for (int c = 0; c < PVE_OBS_W; ++c) rows_cur[(size_t)M.newpos[k] * PVE_OBS_W + c] = rows_new[(size_t)k * PVE_OBS_W + c];
        }
    }
    if constexpr (SRC) {
        /* rows_new[newpos[k]] = this tick's row of k, or (a survivor that was no agent) what rows_cur holds there, as the
         * SRC = false branch leaves it.  In place: newpos increases with k, but a vehicle moves down (removals before it)
         * or up (arrivals on an earlier lane).  A slot a vehicle moves down to was held by a vehicle that moves down or
         * stays, or by a removed one, and one it moves up to by a vehicle that moves up or by a removed one; so one pass
         * over the first kind in increasing k and one over the second in decreasing k read every row before a store can
         * reach it.  Each lane owns one column, so the lanes need no synchronisation. */
        P4_PAR(c, PVE_OBS_W) {
            for (int k0 = 0; k0 < V; k0 += 8) pve4_move_rows<true>(M, rows_new, rows_cur, c, k0, V);
            for (int k0 = V - 1; k0 >= 0; k0 -= 8) pve4_move_rows<false>(M, rows_new, rows_cur, c, k0, V);
        }
        P4_SYNC;      /* a spawn slot below may be a slot read above */
    }
    float *const rows_next = SRC ? rows_new : rows_cur;
    P4_PAR(i, PVE4_NLX) {
        if (M.spawn[i]) {                                                                         /* TIS:395-427 */
            const int np = M.spawn[i] - 1, it = M.spawn_int[i];
            const size_t o = vbase + (size_t)np;
            S.p[o] = P.lane_in + P.L[it]; S.v[o] = P.v0; S.a[o] = 0.0; S.js[o] = 0.0;
            pve_veh_meta mt;
            mt.uid = M.spawn_uid[i];
            mt.packed = ((uint32_t)(PVE_F_CONTROL | (1u << 3) | ((uint32_t)it << 5))) << 24;
            S.meta[o] = mt;
            for (int c = 0; c < PVE_OBS_W; ++c) rows_next[(size_t)np * PVE_OBS_W + c] = 0.f;
        }
    }
    P4_SYNC;
    P4_PAR(t, (int)(PVE_HDR_BYTES / 16)) ((pve_v4 *)(S.hdr + b))[t] = ((const pve_v4 *)&M.h)[t];
    P4_ONE {
        S.n_ctrl[b] = M.h.n_ctrl; S.n_veh[b] = M.h.n_veh;
        if (O.agent_offset) {
            O.agent_offset[b] = (int32_t)obase;
            if (b == P.B - 1) O.agent_offset[P.B] = (int32_t)obase + NA;
        }
        if (O.env_collisions) O.env_collisions[b] = M.misc[P4M_COLL];
        if (O.env_lock) O.env_lock[b] = M.misc[P4M_LOCK];
        if (O.env_removed) O.env_removed[b] = M.misc[P4M_NREM];
        double rs = 0, rq = 0, jk = 0;
        for (int g = 0; g < G; ++g) { const double r = (double)M.rew[g]; rs += r; rq += r * r; if (M.fin_now[M.rowveh[g]]) jk += M.js[M.rowveh[g]]; }
        double *st = S.stats + (size_t)b * PVE_NSTAT;
        st[PVE_STAT_AGENT] += (double)NA; st[PVE_STAT_VEH] += (double)V; st[PVE_STAT_COLL] += (double)M.misc[P4M_COLLAG];
        st[PVE_STAT_LOCK] += (double)M.misc[P4M_LOCK]; st[PVE_STAT_JERK] += jk; st[PVE_STAT_RSUM] += rs; st[PVE_STAT_RSQ] += rq;
        st[PVE_STAT_REMOVED] += (double)M.misc[P4M_NREM]; st[PVE_STAT_STEPS] += 1.0; st[PVE_STAT_Q5U] += (double)M.misc[P4M_Q5U];
    }
}
