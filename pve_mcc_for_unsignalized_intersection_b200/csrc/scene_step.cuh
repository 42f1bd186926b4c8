/*
 * scene_step.cuh -- one tick of one intersection, executed by one CTA.
 *
 * Replaces, for lane_num = 12, the reference's step() x V (traffic_interaction_scene.py
 * "TIS" 1501-1539), scene_update() (TIS:222-376) with get_virtual_distance (TIS:733-803),
 * get_p (TIS:1250-1290), get_state (TIS:1292-1338), virtual_lane_search_closer (TIS:1340-1405),
 * check_lock (TIS:1469-1499), add_new_veh (TIS:378-433) and delete_vehicle() (TIS:435-444).
 *
 * The reference is sequential and order dependent; this file is an order-free reformulation
 * (SURVEY.md section 3.3, Q1-Q6):
 *   Q1  rear-end safety chain      -> two candidate next states per vehicle + a chain of
 *                                     1-bit boolean functions resolved per lane
 *   Q2  stale virtual-lane head    -> (head_lane, head_j) persisted in the header
 *   Q3  neighbour rows             -> this tick's row 0 if the neighbour precedes the ego in
 *                                     (lane, j) order, else last tick's row (ping-pong buffer)
 *   Q4  collision counters         -> hit bit per agent + "earlier hitters" / "all hitters" counts
 *   Q5  reward[-1] overrides       -> resolved per agent after all flags are known
 *   Q6  stable sorts               -> total orders (pos, slot) and (|delta|, rank)
 *
 * All state arithmetic is IEEE float64 with contraction disabled (nvcc -fmad=false), in the
 * reference's association order, so p, v, a, jerk_sum stay bit-identical to the float64
 * reference.  Rewards are float64 too but may use reciprocal multiplies (they are outputs, not
 * state; tolerance 1e-5 relative).
 *
 * The body is written as barrier-separated phases (PVE_FOR_TID / PVE_END_TID).  nvcc compiles
 * it as the CUDA kernel.  tests/emul/ compiles THE SAME SOURCE with g++ as a sequential
 * emulation (each phase looped over tid) so that the CPU-only test tier can check the kernel
 * logic against the oracle.  The emulation is test infrastructure: the product library never
 * contains it.
 */
#pragma once
#include <stddef.h>
#include <math.h>
#include <stdint.h>
#include <string.h>
#ifndef __CUDACC__
#include <assert.h>
#endif

#include "pve_mcc.h"

#ifdef __CUDACC__
#define PVE_DEV __device__ __forceinline__
#define PVE_HD __host__ __device__ __forceinline__
#define PVE_FOR_TID(tid) { const int tid = (int)threadIdx.x;
#ifdef PVE_PHASE_TIMING      /* tools/phase_timing.py only: cycle stamp of every phase boundary, CTA thread 0 */
#define PVE_END_TID } __syncthreads(); if (threadIdx.x == 0 && pve_nstamp < 48) pve_stamp[pve_nstamp++] = clock64();
#define PVE_END_TID_NOSYNC } if (threadIdx.x == 0 && pve_nstamp < 48) pve_stamp[pve_nstamp++] = clock64();
#else
#define PVE_END_TID } __syncthreads();
#define PVE_END_TID_NOSYNC }      /* the next phase reads nothing this one wrote */
#endif
/* After phase G1 the CTA splits: threads [0, NS) ("team") finish the tick with named barrier 1,
 * threads [NS, NT) move the observation rows concurrently and exit.  NS == NT: no split. */
#ifdef PVE_PHASE_TIMING
#define PVE_TEAM_STAMP if (threadIdx.x == 0 && pve_nstamp < 48) pve_stamp[pve_nstamp++] = clock64();
#else
#define PVE_TEAM_STAMP
#endif
#define PVE_FOR_TEAM(tid) { const int tid = (int)threadIdx.x;
#define PVE_END_TEAM } pve_team_sync<NS, NT>(); PVE_TEAM_STAMP
#define PVE_ATOMIC_ADD(ptr, val) atomicAdd((ptr), (val))
#define PVE_RED_ADD(ptr, val) atomicAdd((ptr), (val))   /* result unused: a RED, nothing to wait for */
#define PVE_RESTRICT __restrict__
#else
#define PVE_DEV static inline
#define PVE_HD static inline
#define PVE_FOR_TID(tid) for (int tid = 0; tid < NT; ++tid) {
#define PVE_END_TID }
#define PVE_END_TID_NOSYNC }
#define PVE_FOR_TEAM(tid) for (int tid = 0; tid < NS; ++tid) {
#define PVE_END_TEAM }
static inline int pve_emul_atomic_add(int *p, int v) { int o = *p; *p = o + v; return o; }
#define PVE_ATOMIC_ADD(ptr, val) pve_emul_atomic_add((ptr), (val))
#define PVE_RED_ADD(ptr, val) (*(ptr) += (val))
#define PVE_RESTRICT __restrict__
#endif

#include "arrivals.cuh"

struct alignas(16) pve_v4 { uint32_t x, y, z, w; };
struct alignas(16) pve_d2 { double x, y; };

/* kernel parameters (by value; lives in the constant bank) */
struct PveParams {
    double dt, dt2, vm, vM, am, aM, v0, thr, lane_in, remove_p, lane_cw, abs_am, two_abs_am, aspan;
    double r_abs_am, r_two_abs_am;      /* reciprocals, used only to pre-screen the rear-end test (phase B) */
    double lane_len[3];
    double spawn_p[3];
    double vd_a1[2][4], vd_a2[2][4], vd_b[2][4];
    double rot_cos[4], rot_sin[4];
    float f_cw, f_thr, f_len[3], f_rq[3];   /* float copies for the collision pre-screen; f_rq[m] = 3.141593 / 2 / lane_len[m] */
    float f_rc[4], f_rs[4];
    int8_t l2l[PVE_NLANE][4];      /* lane2lane, TIS:153-166 */
    int8_t rev_dir[PVE_NLANE][4];  /* directions d whose lane2lane[d] contains this lane ... */
    int8_t rev_k[PVE_NLANE][4];    /* ... and its position k there */
    int32_t B, VC, AC, K;
    int32_t zero_unctl, pad_;      /* pve_config.zero_uncontrolled */
    int64_t out_cap;
};

struct PveState {
    pve_env_header *hdr;
    double *p, *v, *a, *js;
    pve_veh_meta *meta;
    float *row0[2];           /* ping-pong: [phase] is read, [phase ^ 1] is written */
    int32_t *n_ctrl, *n_veh;  /* [B] this tick's counts (read by every later CTA of the group) */
    int32_t *n_ctrl_next;     /* [B] next tick's counts: separate buffer, CTAs finish in any order */
    double *stats;            /* [B][PVE_NSTAT] running per-intersection statistics */
    /* Row offsets of the dense outputs without a scan kernel: intersections are grouped by 128;
     * gs_read[g] = agents of group g this tick.  A CTA's first row = sum of the earlier groups + the
     * earlier members of its own group (n_ctrl, written last tick).  At its end every CTA adds its
     * next-tick count to gs_acc; gs_zero is cleared for the tick after (three rotating buffers). */
    const int32_t *gs_read;
    int32_t *gs_acc, *gs_zero;
    void *dbg;                /* tools/phase_timing.py builds only: [B][48] cycle stamps */
    const int32_t *order;     /* CTA index -> intersection, busiest first (refreshed every few ticks), or null */
    /* Two kernels per tick (pve_mcc.cu, "dual mode"): intersections that fit the small capacity class run in small
     * CTAs, the few others in CTAs of the handle's full class.  Every CTA classifies its intersection for the NEXT
     * tick when it ends (klass_next, big_list_next); the three counters rotate like the group sums. */
    const uint8_t *klass;     /* [B] 1: this tick the intersection belongs to the big kernel; null: single kernel */
    uint8_t *klass_next;
    const int32_t *big_list;  /* intersections of the big kernel this tick, big_cnt[0] of them */
    int32_t *big_list_next;
    const int32_t *big_cnt;
    int32_t *big_cnt_next, *big_cnt_zero;
    int32_t small_vc, small_ac;
};

enum { PVE_STAT_AGENT = 0, PVE_STAT_VEH, PVE_STAT_COLL, PVE_STAT_LOCK, PVE_STAT_JERK, PVE_STAT_RSUM,
       PVE_STAT_RSQ, PVE_STAT_REMOVED, PVE_STAT_STEPS, PVE_STAT_Q5U, PVE_NSTAT };

/* ---------------------------------------------------------------------------------------------
 * shared-memory layout: compile-time offsets for a capacity class (VC vehicle slots, AC agents,
 * EC = 5*AC virtual-lane entries).  Regions R1 and R2 are reused along the tick:
 *   R1: step candidates (phases A-C) -> unsorted virtual-lane entries (E-F) -> row 0 of every agent (G1-M)
 *   R2: sorted virtual lanes (F-I)
 * (per-row cp.async.bulk stores were measured and rejected: ~225 tiny TMA operations per
 * intersection saturate the copy engine; see DESIGN.md)
 * ------------------------------------------------------------------------------------------- */
template <int VC, int AC>
struct PveLayout {
    static constexpr uint32_t a16(uint32_t x) { return (x + 15u) & ~15u; }
    static constexpr uint32_t mx(uint32_t a, uint32_t b) { return a > b ? a : b; }
    static constexpr int EC = 5 * AC + 16;              /* each direction's segment is padded to an even length */
    static constexpr int SC = EC + 12 * PVE_NLANE;      /* sorted lists: 6 sentinels below and above each direction's */
    static constexpr uint32_t HDR = 0;
    static constexpr uint32_t SP = a16(PVE_HDR_BYTES);
    static constexpr uint32_t SV = SP + 8 * VC;
    static constexpr uint32_t SA = SV + 8 * VC;
    static constexpr uint32_t SJS = SA + 8 * VC;
    static constexpr uint32_t R1 = a16(SJS + 8 * VC);
    static constexpr uint32_t CTA0 = R1, CP0 = CTA0 + 8 * VC, CV0 = CP0 + 8 * VC,
                              CP1 = CV0 + 8 * VC, CV1 = CP1 + 8 * VC;
    static constexpr uint32_t EPOS = R1, EIDX = EPOS + 8 * EC;
    static constexpr uint32_t ROW0 = R1;                          /* f32[AC + 1][28]; row AC is all zero */
    static constexpr uint32_t R1_BYTES = mx(mx(40 * VC, a16(10 * EC)), 112 * (AC + 1));
    static constexpr uint32_t R2 = a16(R1 + R1_BYTES);
    static constexpr uint32_t SPOS = R2, SIDX = SPOS + 8 * SC;
    static constexpr uint32_t R2_BYTES = a16(10 * SC);
    static constexpr uint32_t XY = a16(R2 + R2_BYTES);               /* world coordinates of the agents (G1-G3) */
    static constexpr uint32_t DSUM = XY + 16 * AC;
    static constexpr uint32_t REW = DSUM + 8 * 8;
    static constexpr uint32_t SUID = REW + 4 * AC;
    static constexpr uint32_t SPK = SUID + 4 * VC;
    static constexpr uint32_t INCB = SPK + 4 * VC;
    static constexpr uint32_t INCT = INCB + 4 * AC;
    static constexpr uint32_t CPV = INCT + 4 * AC;
    static constexpr uint32_t LANE_OFF = CPV + 4 * AC;           /* int[16] */
    static constexpr uint32_t VL_BASE = LANE_OFF + 64;           /* int[16] */
    static constexpr uint32_t AFIRST = VL_BASE + 64;             /* int[16]: first agent of each lane */
    static constexpr uint32_t SEG = AFIRST + 64;                 /* u16[48]: offset of source lane q inside direction d's segment */
    static constexpr uint32_t MISC = SEG + 96;                   /* int[56] */
    static constexpr uint32_t WSUM = MISC + 224;                 /* int[96]: [0,32) scans, [32,64) chain, [64,80) first row; 16 warps */
    static constexpr uint32_t ACNT = WSUM + 384;                 /* u16[VC+2] */
    static constexpr uint32_t SURV = ACNT + a16(2 * (VC + 2));
    static constexpr uint32_t VIDX = SURV + a16(2 * (VC + 2));
    static constexpr uint32_t ARANK = VIDX + 2 * AC;
    static constexpr uint32_t HDRA = ARANK + 2 * AC;
    static constexpr uint32_t NN0 = HDRA + 2 * AC;
    static constexpr uint32_t SRC = NN0 + 2 * AC;                /* u16[AC][7] gather codes */
    static constexpr uint32_t HEADK = a16(SRC + 14 * AC);        /* i16[16] */
    static constexpr uint32_t TIE = HEADK + 32;                  /* u8[16]: direction d has entries at equal positions */
    static constexpr uint32_t LANE_OF = TIE + 16;
    static constexpr uint32_t FBITS = LANE_OF + VC;
    static constexpr uint32_t SSEL = FBITS + VC;
    static constexpr uint32_t DEL = SSEL + VC;
    static constexpr uint32_t SLOCK = DEL + VC;
    static constexpr uint32_t CTL0 = SLOCK + VC;
    static constexpr uint32_t SLOCKA = CTL0 + VC;
    static constexpr uint32_t HIT = SLOCKA + VC;
    static constexpr uint32_t Q5 = HIT + AC;
    static constexpr uint32_t FIN5 = Q5 + AC;
    static constexpr uint32_t STATUS = FIN5 + AC;
    static constexpr uint32_t EDIR = STATUS + AC;                /* u8[EC] direction of each unsorted entry */
    static constexpr uint32_t BYTES = a16(EDIR + EC);
    static_assert(VC % 16 == 0 && AC % 16 == 0 && AC <= VC && VC <= 1024, "capacity class");
};

enum { M_V = 0, M_NREM, M_PASSED, M_COLL, M_LOCK, M_NCTRL, M_Q5U, M_PSTEP, M_COLLAG, M_IDSEQ0,
       M_SPAWN0 /* 12 */, M_SPREF0 = M_SPAWN0 + 12 /* 13 */, M_NEXT0 = M_SPREF0 + 13 /* 12 */,
       M_COUNT = M_NEXT0 + 12 };
static_assert(M_COUNT <= 56, "misc block");

/* gather codes of the 7 observation rows of an agent: the low 15 bits are the first 16-byte piece of
 * the source row (7 pieces per row), bit 15 clear -> in the shared-memory row table (this tick's row 0
 * of an agent; row AC is the zero row of an absent neighbour, TIS:1335), bit 15 set -> in last tick's
 * stored rows of this intersection (indexed by vehicle slot). */
#define PVE_SRC_PREV 0x8000u
#define PVE_ROW_BYTES (PVE_OBS_W * 4)
#define PVE_INF (__builtin_huge_val())

PVE_DEV void pve_prefetch_l2(const void *p) {
#ifdef __CUDACC__
    asm volatile("prefetch.global.L2 [%0];" :: "l"(p));
#else
    (void)p;
#endif
}

PVE_DEV uint32_t pve_fbits(float f) { uint32_t u; memcpy(&u, &f, sizeof u); return u; }
PVE_DEV pve_v4 pve_pack4(float a, float b, float c, float d) {
    pve_v4 r; r.x = pve_fbits(a); r.y = pve_fbits(b); r.z = pve_fbits(c); r.w = pve_fbits(d); return r;
}
/* byte q (0..11) of the 12-byte little-endian array {w0, w1, w2} */
PVE_DEV uint32_t pve_byte12(uint32_t w0, uint32_t w1, uint32_t w2, int q) {
    const uint32_t w = (q < 4) ? w0 : (q < 8 ? w1 : w2);
    return (w >> ((q & 3) * 8)) & 0xFFu;
}
/* number of bytes of x that are <= the corresponding byte of y (unsigned) */
PVE_DEV int pve_count_le4(uint32_t x, uint32_t y) {
#ifdef __CUDACC__
    return __popc(__vcmpleu4(x, y)) >> 3;
#else
    int c = 0;
    for (int q = 0; q < 4; ++q) c += ((x >> (8 * q)) & 0xFFu) <= ((y >> (8 * q)) & 0xFFu);
    return c;
#endif
}
/* 1 if x < 0 else 0 (x is a difference of two finite doubles: a - b < 0 <=> a < b, and a - b is
 * +0 exactly when a == b) */
PVE_DEV uint32_t pve_isneg(double x) {
#ifdef __CUDACC__
    return (uint32_t)__double2hiint(x) >> 31;
#else
    uint64_t u; memcpy(&u, &x, sizeof u); return (uint32_t)(u >> 63);
#endif
}
/* ---------------------------------------------------------------------------------------------
 * block collectives.  Device: warp ballot / shuffle + one smem exchange.  Host emulation:
 * sequential loops over the same shared arrays.
 * ------------------------------------------------------------------------------------------- */
/* out[k] = number of set flags before k (k = 0..n), i.e. an exclusive scan; out[n] = total, which is
 * also returned to every thread.  This is the stream-compaction index used for agent numbering and
 * for vehicle removal.  NO trailing barrier: thread t may read the out[k] it wrote itself
 * (k = t, t + NT, ...) right away; the caller's next phase boundary publishes the rest. */
#ifdef __CUDACC__
template <int NTH, int NTOT>
PVE_DEV void pve_team_sync() {
    if (NTH == NTOT) __syncthreads();
    else asm volatile("bar.sync 1, %0;" :: "n"(NTH) : "memory");
}
#endif
template <int NT, int NTOT = NT>
PVE_DEV int pve_block_excl_scan(const uint8_t *flag, uint16_t *out, int n, int32_t *wsum) {
#ifdef __CUDACC__
    const int tid = (int)threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = NT / 32;
    int carry = 0;
#pragma unroll 1
    for (int base = 0; base < n; base += NT) {
        const int k = base + tid;
        const int f = (k < n) ? (flag[k] != 0) : 0;
        const unsigned bal = __ballot_sync(0xffffffffu, f);
        const int wp = __popc(bal & ((1u << lane) - 1u));
        int32_t *ws = wsum + ((base / NT) & 1) * NW;      /* double-buffered: one barrier per chunk */
        if (lane == 0) ws[warp] = __popc(bal);
        pve_team_sync<NT, NTOT>();
        int woff = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < NW; ++w) { const int c = ws[w]; woff += (w < warp) ? c : 0; tot += c; }
        if (k < n) out[k] = (uint16_t)(carry + woff + wp);
        carry += tot;
    }
    if (tid == 0) out[n] = (uint16_t)carry;
    return carry;
#else
    (void)wsum;
    int c = 0;
    for (int k = 0; k < n; ++k) { out[k] = (uint16_t)c; c += (flag[k] != 0); }
    out[n] = (uint16_t)c;
    return c;
#endif
}

/* Q1 chain: s_k = F_k(s_{k-1}) with F_k a boolean function of one boolean, stored as two bits
 * (bit x = F_k(x)).  Function composition is associative, so the chain over the dense vehicle
 * order is an inclusive scan; a lane's front vehicle has the constant function 0, which restarts
 * the chain, so no segmentation is needed.  Thread t writes sel[k] only for its own k. */
PVE_HD uint32_t pve_compose(uint32_t later, uint32_t earlier) {      /* (later o earlier) */
    return ((later >> (earlier & 1u)) & 1u) | (((later >> ((earlier >> 1) & 1u)) & 1u) << 1);
}
template <int NT>
PVE_DEV void pve_resolve_chain(const uint8_t *fbits, uint8_t *sel, int n, int32_t *ws16) {
#ifdef __CUDACC__
    const int tid = (int)threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = NT / 32;
    uint32_t carry = 0;                                   /* state entering the chunk */
#pragma unroll 1
    for (int base = 0; base < n; base += NT) {
        const int k = base + tid;
        uint32_t g = (k < n) ? (uint32_t)fbits[k] : 2u;   /* 2 = identity */
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, g, d);
            if (lane >= d) g = pve_compose(g, t);
        }
        int32_t *ws = ws16 + ((base / NT) & 1) * NW;
        if (lane == 31) ws[warp] = (int32_t)g;
        __syncthreads();
        uint32_t s_in = carry, s_all = carry;
#pragma unroll
        for (int w = 0; w < NW; ++w) {
            const uint32_t tw = (uint32_t)ws[w];
            s_all = (tw >> s_all) & 1u;
            if (w < warp) s_in = s_all;
        }
        if (k < n) sel[k] = (uint8_t)((g >> s_in) & 1u);
        carry = s_all;
    }
#else
    (void)ws16;
    uint32_t st = 0;
    for (int k = 0; k < n; ++k) { st = ((uint32_t)fbits[k] >> st) & 1u; sel[k] = (uint8_t)st; }
#endif
}

/* first output row of intersection b (see PveState::gs_read); result returned to every thread */
#define PVE_GROUP_SHIFT 7
struct PveRowPart { int g, n; };
template <int NT>
PVE_DEV PveRowPart pve_first_row_part(const PveState &S, int b) {      /* this thread's share: loads issued early, */
    PveRowPart r; r.g = 0; r.n = 0;                                     /* nothing consumed before pve_first_row    */
#ifdef __CUDACC__
    const int tid = (int)threadIdx.x;
    const int i0 = (b >> PVE_GROUP_SHIFT) << PVE_GROUP_SHIFT;
    if (tid < (b >> PVE_GROUP_SHIFT)) r.g = S.gs_read[tid];
    if (i0 + tid < b) r.n = S.n_ctrl[i0 + tid];
#else
    (void)S; (void)b;
#endif
    return r;
}
template <int NT>
PVE_DEV int pve_first_row(const PveState &S, int b, PveRowPart rp, int32_t *ws) {
#ifdef __CUDACC__
    const int tid = (int)threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int part = rp.g + rp.n;
#pragma unroll 1
    for (int i = tid + NT; i < (b >> PVE_GROUP_SHIFT); i += NT) part += S.gs_read[i];          /* B > 128 * NT only */
#pragma unroll 1
    for (int i = ((b >> PVE_GROUP_SHIFT) << PVE_GROUP_SHIFT) + tid + NT; i < b; i += NT) part += S.n_ctrl[i];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) part += __shfl_xor_sync(0xffffffffu, part, d);
    if (lane == 0) ws[warp] = part;
    __syncthreads();
    int tot = 0;
#pragma unroll
    for (int w = 0; w < NT / 32; ++w) tot += ws[w];
    return tot;
#else
    (void)ws; (void)rp;
    int tot = 0;
    for (int i = 0; i < (b >> PVE_GROUP_SHIFT); ++i) tot += S.gs_read[i];
    for (int i = ((b >> PVE_GROUP_SHIFT) << PVE_GROUP_SHIFT); i < b; ++i) tot += S.n_ctrl[i];
    return tot;
#endif
}

/* statistics of the tick, computed by warp 0 only (no barrier): sum r, sum r^2, sum of jerk_sum of the agents
 * that finished this tick (TIS:358) */
template <int NT>
PVE_DEV void pve_warp0_sums(const float *x, const uint8_t *fin, const double *js, const uint16_t *vidx, int n, double *out3) {
#ifdef __CUDACC__
    const int tid = (int)threadIdx.x;
    if (tid < 32) {
        double s0 = 0, s1 = 0, s2 = 0;
#pragma unroll 1
        for (int k = tid; k < n; k += 32) {
            const double r = (double)x[k]; s0 += r; s1 += r * r;
            if (fin[k]) s2 += js[vidx[k]];
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            s0 += __shfl_xor_sync(0xffffffffu, s0, d);
            s1 += __shfl_xor_sync(0xffffffffu, s1, d);
            s2 += __shfl_xor_sync(0xffffffffu, s2, d);
        }
        if (tid == 0) { out3[0] = s0; out3[1] = s1; out3[2] = s2; }
        __syncwarp();                                    /* lanes of warp 0 read out3 next (phase K) */
    }
#else
    double a0 = 0, a1 = 0, a2 = 0;
    for (int k = 0; k < n; ++k) { const double r = (double)x[k]; a0 += r; a1 += r * r; if (fin[k]) a2 += js[vidx[k]]; }
    out3[0] = a0; out3[1] = a1; out3[2] = a2;
#endif
}

/* vir_dis of agent t (TIS:1349-1354): gap to the entry just ahead in its own virtual lane, 100 for the head.
 * aidx[t] = index of the agent's entry in the sorted lists; the entry below a head is a -inf sentinel */
PVE_DEV double pve_vir_dis(const double *spos, const uint16_t *aidx, int t) {
    const double *const S = spos + aidx[t];
    const double below = S[-1];
    return below == -PVE_INF ? 100.0 : S[0] - below;
}

/* ---------------------------------------------------------------------------------------------
 * Row mover: the 7 x 28 observation of every agent.  Row 0 is the agent's own row, row q+1 is
 * neighbour q's stored row (Q3): this tick's row if that neighbour was processed earlier (shared
 * memory), else last tick's row (state buffer, prefetched to L2 in phase A), or zeros.
 * It runs on the warps that have no work in the agent phases, concurrently with them (see the CTA
 * split after phase G1).
 * ------------------------------------------------------------------------------------------- */
struct PveRowJob {
    int A;
    const uint16_t *srcc;         /* [A][7] gather codes, see PVE_SRC_PREV */
    const float *rows_smem;       /* [AC + 1][28], row AC = zeros */
    const float *rows_prev;       /* last tick's stored rows of this intersection */
    pve_v4 *oblk;                 /* this intersection's observation block or null */
    int zero_row;                 /* index of the all-zero row of rows_smem */
};

template <int NT, int NW>
PVE_DEV void pve_move_rows(const PveRowJob &J, int first_warp) {
    if (J.oblk == nullptr) return;
#ifdef __CUDACC__
    /* The block of an intersection is contiguous: A x 7 rows of 7 16-byte pieces.  Eight lanes share a row
     * (lane & 7 = piece, the eighth lane idles), so a quarter-warp reads one 112-byte row -- seven distinct
     * bank groups, no conflicts whatever rows the four quarters hold -- and a warp stores 448 contiguous
     * bytes.  The row's gather code is read once per row (a broadcast); the source is read from shared
     * memory unless the code says "last tick's buffer", in which case a predicated global load overrides
     * it. */
    const int t = (int)threadIdx.x - first_warp * 32;
    const int piece = t & 7;
    if (piece == 7) return;
    const int n_rows = J.A * PVE_OBS_H;
    constexpr int RSTEP = 4 * NW;                         /* rows taken by the mover warps per step */
    const pve_v4 *PVE_RESTRICT prev = (const pve_v4 *)J.rows_prev + piece;
    const pve_v4 *rows = (const pve_v4 *)J.rows_smem + piece;
    int row = t >> 3;
    pve_v4 *PVE_RESTRICT dst = J.oblk + piece + row * 7;
    const uint16_t *sc = J.srcc + row;
    /* PVE_MOVER_DEPTH rows in flight per lane: about half of the rows come from last tick's buffer (an L2 hit), and the
     * loop pays one such round trip per iteration whatever the depth */
#ifndef PVE_MOVER_DEPTH
#define PVE_MOVER_DEPTH 8
#endif
    constexpr int D = PVE_MOVER_DEPTH;
    const uint32_t rows_sa = (uint32_t)__cvta_generic_to_shared(rows);
#pragma unroll 1
    for (; row < n_rows; row += D * RSTEP, dst += D * RSTEP * 7, sc += D * RSTEP) {
        pve_v4 val[D];
        /* predicated loads written out: left to the compiler, "row in range ? (last tick's buffer ? global : shared)"
         * becomes divergent branches around every load, and the quarters of a warp (different rows) take them apart */
#pragma unroll
        for (int u = 0; u < D; ++u) {
            const bool ok = row + u * RSTEP < n_rows;
            const uint32_t code = ok ? (uint32_t)sc[u * RSTEP] : 0u;
            const uint32_t src = code & 0x7FFFu;
            const uint32_t sel = ok ? (code >> 15) : 2u;              /* 0: shared, 1: global, 2: no row */
            asm volatile("{\n\t.reg .pred pg, ps;\n\t"
                         "setp.eq.u32 pg, %6, 1;\n\t"
                         "setp.eq.u32 ps, %6, 0;\n\t"
                         "@pg ld.global.v4.u32 {%0, %1, %2, %3}, [%4];\n\t"
                         "@ps ld.shared.v4.u32 {%0, %1, %2, %3}, [%5];\n\t}"
                         : "=r"(val[u].x), "=r"(val[u].y), "=r"(val[u].z), "=r"(val[u].w)
                         : "l"(prev + src), "r"(rows_sa + src * 16u), "r"(sel));
        }
#pragma unroll
        for (int u = 0; u < D; ++u)
            if (row + u * RSTEP < n_rows) dst[u * RSTEP * 7] = val[u];
    }
#else
    (void)first_warp;
    for (int it = 0; it < J.A * PVE_OBS_H; ++it) {
        const uint32_t c = J.srcc[it];
        const float *src = ((c & PVE_SRC_PREV) ? J.rows_prev : J.rows_smem) + (size_t)(c & 0x7FFFu) * 4;
        memcpy(J.oblk + (size_t)it * 7, src, PVE_OBS_W * sizeof(float));
    }
#endif
}

/* ---------------------------------------------------------------------------------------------
 * Factored observation (pve_outputs.row0_out / prev_row0 / obs_src; SRC instantiation only): per agent its
 * row 0 of this tick, the row stored for its vehicle when the tick started, and the 7 row codes of its
 * observation translated to agent indices.  A neighbour is always an agent of the same tick (virtual
 * lanes hold agents only, phase E), so a "last tick's row" code (PVE_SRC_PREV | slot * 7) becomes
 * 0x4000 | the neighbour's agent index.  Everything read here is final after phase G1 and no later
 * phase writes it, so either half of a split CTA can do it: the mover warps right after G1 when there
 * are no observation rows to move, the team after phase K otherwise.
 * ------------------------------------------------------------------------------------------- */
struct PveFactJob {
    int A, V, AC;
    const uint16_t *srcc;         /* [A][7] gather codes */
    const uint16_t *acnt;         /* [V + 1] agent index of each vehicle slot (exclusive scan of the control flags) */
    const uint16_t *vidx;         /* [A] vehicle slot of each agent */
    const float *rows_smem;       /* [AC + 1][28] this tick's row 0 of every agent */
    const float *rows_prev;       /* last tick's stored rows of this intersection */
    pve_v4 *row0_out, *prev_out;  /* this intersection's first row of pve_outputs.row0_out / prev_row0, or null */
    pve_v4 *src_out;              /* ... of pve_outputs.obs_src */
};

PVE_DEV void pve_write_factored(const PveFactJob &J, int t, int nthreads) {
    if (J.src_out == nullptr) return;
#pragma unroll 1
    for (int it = t; it < J.A * 8; it += nthreads) {
        const int g = it >> 3, q = it & 7;
        if (q < 7) {                       /* 16-byte piece q of both rows: a warp stores 4 rows x 7 pieces contiguously */
            J.row0_out[g * 7 + q] = ((const pve_v4 *)(J.rows_smem + (size_t)g * PVE_OBS_W))[q];
            J.prev_out[g * 7 + q] = ((const pve_v4 *)(J.rows_prev + (size_t)J.vidx[g] * PVE_OBS_W))[q];
        } else {
            uint32_t w4[4];
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                const uint32_t c = r < PVE_OBS_H ? J.srcc[g * 7 + r] : (uint32_t)(J.AC * 7);
                uint32_t v;
                if (c == (uint32_t)(J.AC * 7)) v = 0xFFFFu;                                 /* the zero row */
                else if (c & PVE_SRC_PREV) {
                    const int kn = (int)((c & 0x7FFFu) / 7u);
#ifndef __CUDACC__
                    /* the premise of the contract: the neighbour is an agent of this tick */
                    assert(kn < J.V && J.acnt[kn + 1] == J.acnt[kn] + 1 && J.acnt[kn] < J.A);
#endif
                    v = 0x4000u | J.acnt[kn];
                } else v = c / 7u;
                if (r & 1) w4[r >> 1] |= v << 16; else w4[r >> 1] = v;
            }
            pve_v4 s; s.x = w4[0]; s.y = w4[1]; s.z = w4[2]; s.w = w4[3];
            J.src_out[g] = s;
        }
    }
}

/* ---------------------------------------------------------------------------------------------
 * TIS:1250-1290 get_p for lane_num = 12 (yaw is never read by the caller)
 * ------------------------------------------------------------------------------------------- */
PVE_DEV void pve_world_xy(const PveParams &P, double p, int lane, double *x, double *y) {
    const double cw = P.lane_cw;
    const int m = lane % 3;
    double tx, ty;
    if (m == 1) {
        tx = p - 6 * cw; ty = 3 * cw;                                           /* TIS:1270 */
    } else {
        const double L = P.lane_len[m];
        if (p > L) {
            tx = p - L + 6 * cw; ty = (m == 0) ? cw : 5 * cw;                   /* TIS:1256, 1274 */
        } else if (p > 0) {
            const double r_a = (L - p) / L * 3.141593 / 2;                      /* TIS:1259, 1277 */
            double sn, cs;
#ifdef __CUDACC__
            sincos(r_a, &sn, &cs);
#else
            sn = sin(r_a); cs = cos(r_a);
#endif
            if (m == 0) { tx = 6 * cw - (7 * cw) * sn; ty = -6 * cw + (7 * cw) * cs; }   /* TIS:1262-1263 */
            else        { tx = 6 * cw + (-cw) * sn;    ty = 6 * cw + (-cw) * cs; }       /* TIS:1281-1282 */
        } else if (m == 0) {
            tx = -cw; ty = -6 * cw + p;                                         /* TIS:1267 */
        } else {
            tx = 5 * cw; ty = 6 * cw - p;                                       /* TIS:1286 */
        }
    }
    const double c = P.rot_cos[lane / 3], s = P.rot_sin[lane / 3];              /* TIS:1251 */
    *x = tx * c - ty * s;                                                       /* TIS:1287 */
    *y = ty * c + tx * s;                                                       /* TIS:1288 */
}

/* The same in float32 (sin / cos by the special-function unit): a pre-screen for the collision test.  The error of a
 * coordinate is below 1e-4 m (|coordinates| < 200 m, |sin| error 5e-7 on a radius of 26 m; the two sides of every
 * branch of get_p meet continuously, so a branch taken differently in float32 costs no more than that); phase G3
 * repeats the test in float64 (pve_world_xy) whenever the float32 distance is within PVE_XY_MARGIN of the threshold,
 * so every decision is the float64 one. */
#define PVE_XY_MARGIN 0.02f
PVE_DEV void pve_world_xy_f32(const PveParams &P, double p, int lane, float *x, float *y) {
    const float cw = P.f_cw, pf = (float)p;
    const int m = lane % 3;
    float tx, ty;
    if (m == 1) {
        tx = pf - 6 * cw; ty = 3 * cw;
    } else {
        const float L = P.f_len[m];
        if (pf > L) {
            tx = pf - L + 6 * cw; ty = (m == 0) ? cw : 5 * cw;
        } else if (pf > 0) {
            const float r_a = (L - pf) * P.f_rq[m];
            float sn, cs;
#ifdef __CUDACC__
            __sincosf(r_a, &sn, &cs);
#else
            sn = sinf(r_a); cs = cosf(r_a);
#endif
            if (m == 0) { tx = 6 * cw - (7 * cw) * sn; ty = -6 * cw + (7 * cw) * cs; }
            else        { tx = 6 * cw - cw * sn;       ty = 6 * cw - cw * cs; }
        } else if (m == 0) {
            tx = -cw; ty = -6 * cw + pf;
        } else {
            tx = 5 * cw; ty = 6 * cw - pf;
        }
    }
    const float c = P.f_rc[lane / 3], s = P.f_rs[lane / 3];
    *x = tx * c - ty * s;
    *y = ty * c + tx * s;
}
/* the exact test of phase G3 for the rare pair the pre-screen cannot decide (a rolled loop: one copy of the float64
 * geometry in the instruction stream, in a branch that is almost never fetched) */
PVE_DEV bool pve_collide_exact(const PveParams &P, double p0, int lane0, double p1, int lane1) {
    double x[2], y[2];
#pragma unroll 1
    for (int w = 0; w < 2; ++w) pve_world_xy(P, w ? p1 : p0, w ? lane1 : lane0, &x[w], &y[w]);
    const double dx = x[1] - x[0], dy = y[1] - y[0];
    return sqrt(dx * dx + dy * dy) < P.thr;                                      /* TIS:322-334 */
}

/* ---------------------------------------------------------------------------------------------
 * TIS:293-320 reward of an agent: p, v, jerk/dt of the ego; vd0, v0 = virtual position and speed of its
 * nearest neighbour (has_nb false: none)
 * ------------------------------------------------------------------------------------------- */
PVE_DEV float pve_reward(double vm, double aspan, double p, double v, double jr, bool has_nb, double vd0, double v0) {
    /* The three transcendental terms are evaluated unconditionally on safe arguments and selected afterwards: in a
     * warp some agent needs each of them anyway, and without branches their dependent chains (division -> exp ->
     * division; log) overlap instead of running one after the other. */
    const double gap = p - vd0;
    const double d_raw = fabs(gap);                                              /* TIS:300 */
    const bool near = has_nb && d_raw != 0;
    const double t_distance = near ? gap / (v - v0 + 0.0001) : 2.0;              /* TIS:304 (default TIS:293) */
    const double d_distance = has_nb ? d_raw : 10.0;                             /* TIS:300 (default TIS:294) */
    const bool use_t = 0 < t_distance && t_distance < 4;
    const bool use_d = d_distance < 10;
    /* 1 / tanh(-t / 4) = -(1 + 2 / (exp(t / 2) - 1)) for t in (0, 4) */
    const double e1 = exp((use_t ? t_distance : 2.0) * 0.5) - 1.0;
    const double term_t = -(1.0 + 2.0 / e1);                                     /* TIS:314 */
    const double x = (use_d ? d_distance : 5.0) * 0.1, x2 = x * x;
    const double term_d = log(x2 * x2 * x + 0.00001);                            /* TIS:318 */
    double r_ = use_t ? term_t : 0.0;
    r_ -= jr * jr * (3.0 / 3600.0);                                              /* TIS:316 */
    r_ += use_d ? term_d : 0.0;
    r_ += (v - vm) * (2.0 / aspan);                                              /* TIS:319 */
    return (float)fmin(20.0, fmax(-20.0, r_));                                   /* TIS:320 */
}

/* ---------------------------------------------------------------------------------------------
 * one tick of intersection b
 * ------------------------------------------------------------------------------------------- */
/* SRC: also write pve_outputs.nbr_src.  A template flag, not a run-time test: with the code present but switched off
 * the default kernel measured 2-4 % slower (different register allocation), so it exists in its own instantiation.
 * POI: the arrivals come from the Poisson stream (arrivals.cuh, `arr` is a PvePoisson) instead of the spawn table
 * (`arr` is the table); a template flag for the same reason. */
template <int NT, int VC, int AC, bool SRC = false, bool POI = false>
PVE_DEV void pve_step_block(const PveParams &P, const PveState &S, const pve_outputs &O,
                            const typename PveArrivalsT<POI>::type arr, const float *PVE_RESTRICT actions,
                            const int phase, const int b, unsigned char *smem, const uint8_t *skip_class) {
    typedef PveLayout<VC, AC> L;
    /* after phase G1 threads [0, NS) ("team") finish the tick, threads [NS, NT) ("movers") evaluate the rewards and
     * move the observation rows; NS == NT: no split */
    constexpr int NS = (NT >= 128) ? NT / 2 : (NT == 96 ? 64 : NT);      /* 96: two team warps, one mover warp */
    pve_env_header *const hdr = (pve_env_header *)(smem + L::HDR);
    double *const sp = (double *)(smem + L::SP), *const sv = (double *)(smem + L::SV);
    double *const sa = (double *)(smem + L::SA);
    double *const sjs = (double *)(smem + L::SJS);
    double *const cta0 = (double *)(smem + L::CTA0);
    double *const cp0 = (double *)(smem + L::CP0), *const cv0 = (double *)(smem + L::CV0);
    double *const cp1 = (double *)(smem + L::CP1), *const cv1 = (double *)(smem + L::CV1);
    double *const epos = (double *)(smem + L::EPOS), *const spos = (double *)(smem + L::SPOS);
    uint16_t *const eidx = (uint16_t *)(smem + L::EIDX), *const sidx = (uint16_t *)(smem + L::SIDX);
    float *const row0 = (float *)(smem + L::ROW0);
    float *const xyf = (float *)(smem + L::XY);              /* float2[AC], phases G1-G3 */
    double *const vdis = (double *)(smem + L::XY), *const rsort = vdis + AC;   /* phases H-J: vir_dis of every agent, sorted ring distances */
    double *const dsum = (double *)(smem + L::DSUM);
    float *const rew = (float *)(smem + L::REW);
    int32_t *const suid = (int32_t *)(smem + L::SUID);
    uint32_t *const spk = (uint32_t *)(smem + L::SPK);
    int32_t *const incb = (int32_t *)(smem + L::INCB), *const inct = (int32_t *)(smem + L::INCT);
    int32_t *const cpv = (int32_t *)(smem + L::CPV);
    int32_t *const lane_off = (int32_t *)(smem + L::LANE_OFF), *const vl_base = (int32_t *)(smem + L::VL_BASE);
    int32_t *const afirst = (int32_t *)(smem + L::AFIRST), *const misc = (int32_t *)(smem + L::MISC);
    uint16_t *const seg = (uint16_t *)(smem + L::SEG);
    int32_t *const wsum = (int32_t *)(smem + L::WSUM);
    uint16_t *const acnt = (uint16_t *)(smem + L::ACNT), *const surv = (uint16_t *)(smem + L::SURV);
    uint16_t *const vidx = (uint16_t *)(smem + L::VIDX), *const arank = (uint16_t *)(smem + L::ARANK);
    int16_t *const hdra = (int16_t *)(smem + L::HDRA);
    uint16_t *const nn0 = (uint16_t *)(smem + L::NN0), *const srcc = (uint16_t *)(smem + L::SRC);
    int16_t *const headk = (int16_t *)(smem + L::HEADK);
    uint8_t *const tie = smem + L::TIE;
    uint8_t *const lane_of = smem + L::LANE_OF, *const fbits = smem + L::FBITS, *const ssel = smem + L::SSEL;
    uint8_t *const del = smem + L::DEL, *const slock = smem + L::SLOCK, *const ctl0 = smem + L::CTL0;
    int8_t *const slocka = (int8_t *)(smem + L::SLOCKA);
    uint8_t *const hit = smem + L::HIT, *const q5 = smem + L::Q5, *const fin5 = smem + L::FIN5;
    uint8_t *const status = smem + L::STATUS, *const edir = smem + L::EDIR;

    const size_t vbase = (size_t)b * (size_t)P.VC;      /* P.VC: slots per intersection in HBM; VC: slots this kernel stages */
#if defined(PVE_PHASE_TIMING) && defined(__CUDACC__)
    long long pve_stamp[48];
    int pve_nstamp = 0;
    unsigned long long pve_gt0 = 0;
    if (threadIdx.x == 0) {
        pve_stamp[pve_nstamp++] = clock64();
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(pve_gt0));
    }
#endif

    const PveRowPart row_part = pve_first_row_part<NT>(S, b);       /* loads in flight while the header arrives */
    const float *const row0_prev_base = (phase ? S.row0[1] : S.row0[0]) + vbase * PVE_OBS_W;
    float *const row0_next = (phase ? S.row0[0] : S.row0[1]) + vbase * PVE_OBS_W;

    /* ---- A: header -> shared; load vehicles, both candidate next states (Q1).  Nothing here waits
     *         for another thread: every thread reads the 36 bytes of lane lengths and virtual-lane
     *         heads straight from the header in global memory and finds its own (lane, j) in registers,
     *         while the state of vehicle slot `tid` is already on its way (slots >= V are allocated,
     *         their content is ignored) ------------------------------------------------------------ */
    static_assert(offsetof(pve_env_header, lane_n) == 104 && offsetof(pve_env_header, head_lane) == 116
                  && offsetof(pve_env_header, head_j) == 128 && PVE_NLANE == 12, "lane table bytes");
    PVE_FOR_TID(tid)
        const pve_v4 *const gh = (const pve_v4 *)(S.hdr + b);
        uint32_t lw[12];                                     /* header bytes 96..143 */
        { const pve_v4 t0 = gh[6], t1 = gh[7], t2 = gh[8];
          lw[0] = t0.x; lw[1] = t0.y; lw[2] = t0.z; lw[3] = t0.w; lw[4] = t1.x; lw[5] = t1.y; lw[6] = t1.z;
          lw[7] = t1.w; lw[8] = t2.x; lw[9] = t2.y; lw[10] = t2.z; lw[11] = t2.w; }
#define PVE_LW_BYTE(off) ((lw[(off) >> 2] >> (((off) & 3) * 8)) & 0xFFu)
        double p = 0, v = 0, a = 0, js = 0;
        pve_veh_meta mt; mt.uid = 0; mt.packed = 0;
        float actf = 0.f;
        if (tid < VC) {
            p = S.p[vbase + tid]; v = S.v[vbase + tid]; a = S.a[vbase + tid]; js = S.js[vbase + tid];
            mt = S.meta[vbase + tid]; actf = actions[vbase + tid];
        }
        if (skip_class != nullptr && skip_class[b]) return;          /* dual mode: the other kernel's intersection */
        if (tid < PVE_HDR_BYTES / 16) ((pve_v4 *)hdr)[tid] = gh[tid];
#pragma unroll 1
        for (int q = tid + 1; q < M_COUNT; q += NT) misc[q] = 0;                 /* misc[M_V] is written below */
        if (tid < 16) { headk[tid] = -1; tie[tid] = 0; }
        /* lane lengths -> inclusive prefix, one byte per lane (V <= 255; the large classes take 16-bit sums) */
        uint32_t ip0, ip1, ip2, ex0, ex1, ex2;
        int V_;
        if (VC <= 255) {
            ip0 = lw[2]; ip1 = lw[3]; ip2 = lw[4];
            ip0 += ip0 << 8; ip0 += ip0 << 16;
            ip1 += ip1 << 8; ip1 += ip1 << 16;
            ip2 += ip2 << 8; ip2 += ip2 << 16;
            ip1 += (ip0 >> 24) * 0x01010101u;
            ip2 += (ip1 >> 24) * 0x01010101u;
            ex0 = ip0 << 8; ex1 = (ip1 << 8) | (ip0 >> 24); ex2 = (ip2 << 8) | (ip1 >> 24);      /* exclusive prefix */
            V_ = (int)(ip2 >> 24);
            if (tid <= PVE_NLANE) lane_off[tid] = tid < PVE_NLANE ? (int)pve_byte12(ex0, ex1, ex2, tid) : V_;
            if (tid == 0) misc[M_V] = V_;
        } else {
            ip0 = ip1 = ip2 = ex0 = ex1 = ex2 = 0;
            V_ = 0;
#pragma unroll
            for (int q = 0; q < PVE_NLANE; ++q) V_ += (int)PVE_LW_BYTE(8 + q);
            if (tid == 0) {
                int o = 0;
#pragma unroll
                for (int q = 0; q < PVE_NLANE; ++q) { lane_off[q] = o; o += (int)PVE_LW_BYTE(8 + q); }
                lane_off[PVE_NLANE] = o;
                misc[M_V] = o;
            }
        }
#pragma unroll 1
        for (int k = tid; k < V_; k += NT) {
            if (k != tid) {
                p = S.p[vbase + k]; v = S.v[vbase + k]; a = S.a[vbase + k]; js = S.js[vbase + k];
                mt = S.meta[vbase + k]; actf = actions[vbase + k];
            }
            /* lane of slot k: the last lane whose first slot is <= k; and its virtual-lane head */
            int i, off_i, hl, hj;
            if (VC <= 255) {
                const uint32_t kk = (uint32_t)k * 0x01010101u;
                i = pve_count_le4(ip0, kk) + pve_count_le4(ip1, kk) + pve_count_le4(ip2, kk);       /* lanes that end at or before k */
                off_i = (int)pve_byte12(ex0, ex1, ex2, i);
                hl = (int)(int8_t)pve_byte12(lw[5], lw[6], lw[7], i);
                hj = (int)pve_byte12(lw[8], lw[9], lw[10], i);
            } else {
                int o = 0;
                i = 0; off_i = 0;
                hl = (int)(int8_t)PVE_LW_BYTE(20); hj = (int)PVE_LW_BYTE(32);
#pragma unroll
                for (int q = 1; q < PVE_NLANE; ++q) {
                    o += (int)PVE_LW_BYTE(8 + q - 1);
                    if (k >= o) { i = q; off_i = o; hl = (int)(int8_t)PVE_LW_BYTE(20 + q); hj = (int)PVE_LW_BYTE(32 + q); }
                }
            }
            const int j = k - off_i;
            const uint32_t fl = mt.packed >> 24;
            const bool ctrl = (fl & PVE_F_CONTROL) != 0;
            const double act = (P.zero_unctl && !ctrl) ? 0.0 : (double)actf;     /* MAIN:401-405 when asked for */
            const int lock_a = (int)((fl >> 3) & 3u) - 1;
            double ta = fmin(P.aM, fmax(P.am, act));                             /* TIS:1502 */
            if ((fl & PVE_F_LOCK) && lock_a != 0 && p > 70.0) ta = a + (double)lock_a;   /* TIS:1503-1505 */
            const bool forced = (hl == i && hj == j)                             /* TIS:1517 */
                                || (i % 3 == 2);                                /* TIS:1519 */
            const double ta0 = fmin(P.aM, fmax(P.am, forced ? P.aM : ta));       /* TIS:1521 */
            const double ta1 = forced ? P.aM : P.am;                             /* TIS:1516 */
            const double pv = p - v * P.dt;
            double v0n = fmin(P.vM, fmax(v + ta0 * P.dt, P.vm));                 /* TIS:1530 */
            double v1n = fmin(P.vM, fmax(v + ta1 * P.dt, P.vm));
            if (!ctrl) { v0n = P.v0; v1n = P.v0; }                               /* TIS:1535 */
            cta0[k] = ta0;
            cp0[k] = pv - 0.5 * ta0 * P.dt2;                                     /* TIS:1528 */
            cp1[k] = pv - 0.5 * ta1 * P.dt2;
            cv0[k] = v0n; cv1[k] = v1n;
            sp[k] = p; sv[k] = v; sa[k] = a; sjs[k] = js;
            suid[k] = mt.uid; spk[k] = mt.packed;
            if (ctrl) {      /* its stored row will probably be gathered by the row mover: start the HBM fetch now */
                const float *r = row0_prev_base + (size_t)k * PVE_OBS_W;
                pve_prefetch_l2(r); pve_prefetch_l2(r + PVE_OBS_W - 1);
            }
            lane_of[k] = (uint8_t)i;
            ctl0[k] = ctrl ? 1 : 0;
            del[k] = forced ? 1 : 0;        /* borrowed until phase C */
            slock[k] = 0; slocka[k] = 0;
        }
#undef PVE_LW_BYTE
    PVE_END_TID_NOSYNC
    /* row range of this intersection in the dense outputs (one internal barrier, which also publishes A) */
    const int64_t obase = (int64_t)pve_first_row<NT>(S, b, row_part, wsum + 64);
    const int V = misc[M_V];

    /* ---- B: F_k(s) = "rear-end override fires on k if its leader took candidate s" -------- */
    PVE_FOR_TID(tid)
#pragma unroll 1
        for (int k = tid; k < V; k += NT) {
            const int i = lane_of[k];
            int f = 0;
            if (k > lane_off[i] && ctl0[k] && ctl0[k - 1]) {                     /* TIS:1509-1510 */
                const double v = sv[k], p = sp[k];
#pragma unroll
                for (int s = 0; s < 2; ++s) {
                    const double vf = s ? cv1[k - 1] : cv0[k - 1];
                    const double pf = s ? cp1[k - 1] : cp0[k - 1];
                    if (vf < v) {
                        /* TIS:1512-1515 decide p - pf < d_safe.  The two float64 divisions are only needed when the
                         * margin is within 1e-9 of zero: a reciprocal-multiply estimate (error < 1e-12 at these
                         * magnitudes) settles every other case with the same outcome. */
                        const double gap = p - pf, dv2 = v * v - vf * vf, dvm = (v - vf) * P.vm;
                        const double est = v * 0.4 + dv2 * P.r_two_abs_am - dvm * P.r_abs_am;
                        bool fire;
                        if (gap < est - 1.0e-9) fire = true;
                        else if (gap > est + 1.0e-9) fire = false;
                        else fire = gap < v * 0.4 + dv2 / P.two_abs_am - dvm / P.abs_am;
                        if (fire) f |= (1 << s);
                    }
                }
            }
            fbits[k] = (uint8_t)f;
        }
    PVE_END_TID_NOSYNC

    /* ---- B2: resolve the chain (scan of boolean functions; one internal barrier) ------------ */
    pve_resolve_chain<NT>(fbits, ssel, V, wsum + 32);

    /* ---- C: commit kinematics -------------------------------------------------------------- */
    PVE_FOR_TID(tid)
#pragma unroll 1
        for (int k = tid; k < V; k += NT) {
            const int s = ssel[k];
            const double a_new = (s && !del[k]) ? P.am : cta0[k];                /* TIS:1516-1520 */
            del[k] = 0;
            const double jr = (a_new - sa[k]) / P.dt;                            /* TIS:1522, 316, 321 */
            if (ctl0[k]) sjs[k] += fabs(jr);                                     /* TIS:321 */
            sa[k] = a_new;                                                       /* TIS:1523 */
            sp[k] = s ? cp1[k] : cp0[k];
            sv[k] = s ? cv1[k] : cv0[k];
            uint32_t pk = spk[k];
            uint32_t step = pk & 0xFFFFu;
            step = step < 0xFFFFu ? step + 1 : step;                             /* TIS:1533 */
            const uint32_t fl = (pk >> 24) & (PVE_F_CONTROL | PVE_F_FINISH);     /* TIS:1506-1507 */
            spk[k] = (pk & 0x00FF0000u) | step | (fl << 24);
        }
    PVE_END_TID_NOSYNC

    /* ---- agent numbering: controlled at step() time == gets outputs this tick ------------- */
    const int A = pve_block_excl_scan<NT>(ctl0, acnt, V, wsum);           /* == hdr->n_ctrl */
    /* this intersection's block of the dense outputs (null: rows are not emitted) */
    const bool out_ok = obase + A <= P.out_cap && A <= AC;
    pve_v4 *const oblk = (O.obs != nullptr && out_ok) ? (pve_v4 *)O.obs + obase * (PVE_OBS_H * PVE_OBS_W / 4) : nullptr;

    /* ---- D: agent tables (each thread uses only the counts it wrote itself) ---------------- */
    PVE_FOR_TID(tid)
#pragma unroll 1
        for (int k = tid; k < V; k += NT)
            if (ctl0[k]) vidx[acnt[k]] = (uint16_t)k;
#pragma unroll 1
        for (int g = tid; g < A; g += NT) {
            incb[g] = 0; inct[g] = 0; q5[g] = 0; fin5[g] = 0; status[g] = 0; hit[g] = 0;
        }
        /* the sorted lists' region is preset to +inf (an upper bound of what the 12 lists and their sentinels take):
         * whatever phase F does not overwrite is an upper sentinel */
#pragma unroll 1
        for (int e = tid; e < 5 * A + 12 + 12 * PVE_NLANE && e < L::SC; e += NT) spos[e] = PVE_INF;
    PVE_END_TID

    /* ---- D2: the unsorted entries of direction d form one segment: its own agents, then the agents of
     *          its 4 conflicting lanes, each source lane at a fixed offset (seg) so that phase E places every
     *          entry without a reservation; segments are padded to an even length with a +inf entry and the
     *          bases are the exclusive prefix over the 12 lanes (lanes of warp 0) ------------------------- */
    PVE_FOR_TID(tid)
        if (tid < 32) {
#ifdef __CUDACC__
            const int d0 = tid, d1 = tid + 1;
#else
            const int d0 = 0, d1 = (tid == 0) ? PVE_NLANE + 1 : 0;               /* thread 0 walks all lanes */
            int run = 0;
#endif
            for (int d = d0; d < d1; ++d) {
                int o = 0;
                if (d < PVE_NLANE) {
                    afirst[d] = (int)acnt[lane_off[d]];
                    if (hdr->lane_n[d] > 0) {                                    /* TIS:234 */
                        o = (int)acnt[lane_off[d + 1]] - (int)acnt[lane_off[d]];
                        if (d % 3 != 2) {
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                const int Lq = P.l2l[d][q];
                                seg[d * 4 + q] = (uint16_t)o;
                                o += (int)acnt[lane_off[Lq + 1]] - (int)acnt[lane_off[Lq]];
                            }
                        }
                    }
                }
                const int o4 = (o + 1) & ~1;                                     /* even: phase F loads pairs */
#ifdef __CUDACC__
                int incl = o4;
#pragma unroll
                for (int sh = 1; sh < 16; sh <<= 1) {
                    const int t = __shfl_up_sync(0xffffffffu, incl, sh);
                    if (tid >= sh) incl += t;
                }
                const int base = incl - o4;
#else
                const int base = run; run += o4;
#endif
                if (d <= PVE_NLANE) vl_base[d] = base;
                if (o4 != o) { epos[base + o] = PVE_INF; edir[base + o] = 0xFF; }
            }
        }
    PVE_END_TID

    /* ---- E: virtual-lane membership: each agent offers itself to its own lane and to the four lanes it
     *         conflicts with (slot = segment base + source-lane offset + its index among its lane's agents;
     *         an agent that is not a member leaves a +inf entry) --------------------------------------- */
    PVE_FOR_TID(tid)
#pragma unroll 1
        for (int g = tid; g < A; g += NT) {
            const int k = vidx[g];
            const int Lk = lane_of[k];
            const double p = sp[k];
            const int ai = g - afirst[Lk];
            const int e0 = vl_base[Lk] + ai;                                     /* TIS:242-249 */
            epos[e0] = p; eidx[e0] = (uint16_t)k; edir[e0] = (uint8_t)Lk;
            if (Lk % 3 != 2) {
                /* all look-ups first, the stores afterwards: four independent chains instead of four branches */
                int e[4], edv[4];
                double pos[4];
                bool ex[4];
#pragma unroll
                for (int s = 0; s < 4; ++s) {
                    const int dd = P.rev_dir[Lk][s], q = P.rev_k[Lk][s];
                    const int mv = dd % 3;
                    ex[s] = hdr->lane_n[dd] > 0;                                 /* TIS:234 */
                    const double delta = (p - P.vd_a1[mv][q]) + P.vd_a2[mv][q];  /* TIS:733-803 */
                    const bool member = delta > 0;                               /* TIS:259 */
                    pos[s] = member ? P.vd_b[mv][q] + delta : PVE_INF;
                    edv[s] = member ? dd : 0xFF;
                    e[s] = vl_base[dd] + (int)seg[dd * 4 + q] + ai;              /* meaningless unless ex[s] */
                }
#pragma unroll
                for (int s = 0; s < 4; ++s)
                    if (ex[s]) { epos[e[s]] = pos[s]; eidx[e[s]] = (uint16_t)k; edir[e[s]] = (uint8_t)edv[s]; }
            }
        }
    PVE_END_TID

    /* ---- F: stable sort by position (TIS:271) as a rank count on the key (pos, slot).  The sorted list of
     *         direction d lives at spos[vl_base[d] + 12 d + 6 ...] between six -inf and six +inf sentinels,
     *         so that phase G1 reads its twelve candidates without bounds checks.  A segment has an even
     *         number of entries and its non-members are +inf, so the count runs unchecked, two entries per load */
    PVE_FOR_TID(tid)
#pragma unroll 1
        for (int e = tid; e < vl_base[PVE_NLANE]; e += NT) {
            const int d = edir[e];
            if (d != 0xFF) {
                const int base = vl_base[d], n2 = vl_base[d + 1] - base;
                const double pos = epos[e];
                const int idx = eidx[e];
                uint32_t less = 0, greater = 0;
                const pve_d2 *const ep2 = (const pve_d2 *)(epos + base);
#pragma unroll 4
                for (int t = 0; t < n2; t += 2) {
                    const pve_d2 u0 = ep2[t >> 1];
                    less += pve_isneg(u0.x - pos); greater += pve_isneg(pos - u0.x);
                    less += pve_isneg(u0.y - pos); greater += pve_isneg(pos - u0.y);
                }
                int rank = (int)less;
                const int sb = base + 12 * d + 6;
                if (n2 - (int)less - (int)greater > 1) {      /* equal positions keep insertion (slot) order */
#pragma unroll 1
                    for (int t = 0; t < n2; ++t)
                        rank += (epos[base + t] == pos && (int)eidx[base + t] < idx) ? 1 : 0;
                    tie[d] = 1;
                }
                spos[sb + rank] = pos; sidx[sb + rank] = (uint16_t)idx;
                if (lane_of[idx] == d) arank[acnt[idx]] = (uint16_t)(sb + rank);   /* where the agent sits in its own list */
                if (rank == 0) headk[d] = (int16_t)idx;     /* virtual_lane_4[d][0], read by step() (Q2) */
            }
        }
#pragma unroll 1
        for (int q = tid; q < 6 * PVE_NLANE; q += NT) {        /* the lower sentinels */
            const int d = q / 6, w = q - d * 6;
            spos[vl_base[d] + 12 * d + 5 - w] = -PVE_INF;
        }
    PVE_END_TID

    /* ---- G1: per agent: vir_header, six neighbours, row 0, gather codes -------------------- */
    PVE_FOR_TID(tid)
#pragma unroll 1
        for (int g = tid; g < A; g += NT) {
            const int k = vidx[g];
            const int d = lane_of[k];
            const int ax = arank[g];                            /* the ego's entry in the sorted lists (phase F) */
            const double a_old = S.a[vbase + k];                /* last tick's a, still in HBM: jerk of the reward (TIS:316) */
            const double *const S_ = spos + ax;                 /* S_[-r-6 .. -r-1] = -inf, S_[n-r .. n-r+5] = +inf */
            const uint16_t *const SI = sidx + ax;
            const double pe = S_[0];
            /* Six nearest by |delta|, ties to the lower list index (stable sort, TIS:1389).  Only the six
             * entries below and the six above the ego can qualify; both sides are sorted by distance, so the
             * answer is the head of a two-way merge in which the below side wins ties (lower list index).
             * The sentinels make bounds checks unnecessary: an exhausted side has distance +inf. */
            const double dl0 = pe - S_[-1];
            /* vir_header, TIS:1349-1354 (vir_dis: pve_vir_dis, phase I) */
            hdra[g] = (dl0 == PVE_INF) ? (int16_t)-1 : (int16_t)acnt[SI[-1]];
            pve_v4 *const orow = (pve_v4 *)(row0 + (size_t)g * PVE_OBS_W);
            orow[0] = pve_pack4((float)pe, (float)sv[k], (float)sa[k], (float)d);        /* TIS:1336 */
            uint16_t *const sc = srcc + g * 7;
            sc[0] = (uint16_t)(g * 7);
            int nb0 = 0xFFFF, x0 = 0;                          /* nearest neighbour: vehicle slot, list index relative to the ego */
            if (tie[d]) {
                /* entries at equal positions in this list (rare): among equal |delta| below the ego the farther
                 * list index comes first -- resolved with the reference's own outward walk */
                int lo = -1, hi = 1, run_cur = 0, run_end = -1;           /* list indices relative to the ego */
                double run_d = 0;
#pragma unroll 1
                for (int q = 0; q < PVE_NNBR; ++q) {
                    if (run_cur > run_end && S_[lo] != -PVE_INF) {
                        run_end = lo; run_d = fabs(S_[lo] - pe);
                        int x = lo;
                        while (fabs(S_[x - 1] - pe) == run_d) --x;              /* a -inf sentinel ends the run */
                        run_cur = x; lo = x - 1;
                    }
                    const bool has_lo = run_cur <= run_end, has_hi = S_[hi] != PVE_INF;
                    int pick = 0;
                    if (has_lo && (!has_hi || run_d <= fabs(S_[hi] - pe))) pick = run_cur++;
                    else if (has_hi) pick = hi++;
                    if (pick != 0) {
                        const int kn = SI[pick];
                        const double vd = S_[pick];
                        orow[q + 1] = pve_pack4((float)vd, (float)sv[kn], (float)sa[kn], (float)lane_of[kn]);
                        sc[q + 1] = (kn < k) ? (uint16_t)(acnt[kn] * 7) : (uint16_t)(PVE_SRC_PREV | (kn * 7));
                        if (q == 0) { nb0 = kn; x0 = pick; }
                    } else {
                        orow[q + 1] = pve_pack4(0.f, 0.f, 0.f, 0.f);             /* TIS:1334 */
                        sc[q + 1] = (uint16_t)(AC * 7);                          /* the zero row */
                    }
                }
            } else {
                /* the merge itself, rolled (code size: the kernel's instruction stream is fetched once per CTA and does
                 * not fit the instruction cache): the next candidate of each side is kept one step ahead */
                int lo = -1, hi = 1;
                double dlo = dl0, dhi = S_[1] - pe;
#pragma unroll 1
                for (int q = 0; q < PVE_NNBR; ++q) {
                    const bool take_lo = dlo <= dhi;                             /* below wins ties: lower list index */
                    const int x = take_lo ? lo : hi;
                    pve_v4 piece = pve_pack4(0.f, 0.f, 0.f, 0.f);                /* TIS:1334 */
                    uint32_t code = (uint32_t)(AC * 7);                          /* the zero row */
                    if ((take_lo ? dlo : dhi) != PVE_INF) {                      /* else: both sides exhausted */
                        const int kn = SI[x];
                        const double vd = S_[x];
                        piece = pve_pack4((float)vd, (float)sv[kn], (float)sa[kn], (float)lane_of[kn]);          /* TIS:1330 */
                        /* Q3: neighbour already processed this tick -> its new row, else last tick's */
                        code = (kn < k) ? (uint32_t)(acnt[kn] * 7) : (PVE_SRC_PREV | (uint32_t)(kn * 7));
                        if (q == 0) { nb0 = kn; x0 = x; }
                    }
                    orow[q + 1] = piece;
                    sc[q + 1] = (uint16_t)code;
                    if (take_lo) { --lo; dlo = pe - S_[lo]; } else { ++hi; dhi = S_[hi] - pe; }
                }
            }
            nn0[g] = (uint16_t)nb0;
            /* reward (TIS:293-320): everything it needs is in this thread's hands */
            {
                const bool has_nb = nb0 != 0xFFFF;
                const double jr = (sa[k] - a_old) / P.dt;                        /* TIS:1522, 316 */
                rew[g] = pve_reward(P.vm, P.aspan, pe, sv[k], jr, has_nb, S_[x0], has_nb ? sv[nb0] : 0.0);
            }
        }
        if (tid < PVE_OBS_W / 4) ((pve_v4 *)(row0 + (size_t)AC * PVE_OBS_W))[tid] = pve_pack4(0.f, 0.f, 0.f, 0.f);
        /* world positions (TIS:1250-1290) on the threads that have no agent in this phase */
        if (NS < NT && tid >= NS)
#pragma unroll 1
            for (int g = tid - NS; g < A; g += NT - NS) {
                const int k = vidx[g];
                pve_world_xy_f32(P, sp[k], lane_of[k], &xyf[2 * g], &xyf[2 * g + 1]);
            }
    PVE_END_TID

    /* ---- CTA split: the upper half of the CTA moves the observation rows (everything they need is
     *      final after G1) while the lower half ("team") finishes the tick ------------------------ */
    PveRowJob RJ;
    RJ.A = A; RJ.srcc = srcc; RJ.rows_smem = row0; RJ.rows_prev = row0_prev_base; RJ.oblk = oblk; RJ.zero_row = AC;
    PveFactJob FJ;
    if (SRC) {
        const bool fact = O.obs_src != nullptr && out_ok;
        FJ.A = A; FJ.V = V; FJ.AC = AC; FJ.srcc = srcc; FJ.acnt = acnt; FJ.vidx = vidx; FJ.rows_smem = row0;
        FJ.rows_prev = row0_prev_base;
        FJ.row0_out = fact ? (pve_v4 *)O.row0_out + obase * (PVE_OBS_W / 4) : nullptr;
        FJ.prev_out = fact ? (pve_v4 *)O.prev_row0 + obase * (PVE_OBS_W / 4) : nullptr;
        FJ.src_out = fact ? (pve_v4 *)O.obs_src + obase : nullptr;
    }
#ifdef __CUDACC__
    if (NS < NT && (int)threadIdx.x >= NS) {
        pve_move_rows<NT, (NT > NS ? (NT - NS) / 32 : 1)>(RJ, NS / 32);
        if (SRC && oblk == nullptr) pve_write_factored(FJ, (int)threadIdx.x - NS, NT - NS);
#ifdef PVE_PHASE_TIMING
        if ((int)threadIdx.x == NS && S.stats) ((long long *)S.dbg)[(size_t)b * 48 + 47] = clock64();
#endif
        return;
    }
#endif

    /* ---- G2 (no CTA split only): world positions (TIS:1250-1290), which the mover warps otherwise computed
     *          during G1 ---------------------------------------------------------------------------------- */
    if (NS == NT) {
    PVE_FOR_TEAM(tid)
#pragma unroll 1
        for (int g = tid; g < A; g += NS) {
            const int k = vidx[g];
            pve_world_xy_f32(P, sp[k], lane_of[k], &xyf[2 * g], &xyf[2 * g + 1]);
        }
    PVE_END_TEAM
    }

    /* ---- G3: collision test in world space, TIS:322-334 ------------------------------------ */
    PVE_FOR_TEAM(tid)
#pragma unroll 1
        for (int g = tid; g < A; g += NS) {
            const int k0 = nn0[g];
            if (k0 != 0xFFFF) {
                const int g0 = acnt[k0];
                const float dx = xyf[2 * g0] - xyf[2 * g], dy = xyf[2 * g0 + 1] - xyf[2 * g + 1];
                const float dist = sqrtf(dx * dx + dy * dy);
                bool coll = dist < P.f_thr;
                if (fabsf(dist - P.f_thr) < PVE_XY_MARGIN) {                     /* too close to call in float32 */
                    const int k = vidx[g];
                    coll = pve_collide_exact(P, sp[k], lane_of[k], sp[k0], lane_of[k0]);
                }
                if (coll) {
                    hit[g] = 1;
                    PVE_ATOMIC_ADD(&inct[g0], 1);                                /* TIS:334 */
                    if (g < g0) PVE_ATOMIC_ADD(&incb[g0], 1);                    /* Q4 */
                }
            }
        }
    PVE_END_TEAM

    /* ---- H: removal / finish flags for every vehicle, TIS:335-359 ------------------------- */
    PVE_FOR_TEAM(tid)
#pragma unroll 1
        for (int k = tid; k < V; k += NS) {
            const int g = ctl0[k] ? (int)acnt[k] : -1;
            uint32_t pk = spk[k];
            const int prev = (int)((pk >> 16) & 0xFFu);
            const int rep = prev + (g >= 0 ? (int)hit[g] + incb[g] : 0);        /* seen at its turn */
            const int fin = prev + (g >= 0 ? (int)hit[g] + inct[g] : 0);        /* end of tick */
            uint32_t fl = pk >> 24;
            const double p = sp[k];
            if (g >= 0) {
                vdis[g] = pve_vir_dis(spos, arank, g);                           /* TIS:1349-1354; read by the ring members in phase I */
                cpv[g] = rep;                                                    /* TIS:337-339 */
                if (rep > 0) { PVE_ATOMIC_ADD(&misc[M_COLL], rep); PVE_ATOMIC_ADD(&misc[M_COLLAG], 1); }
            }
            if (p < P.remove_p || rep > 0) {                                     /* TIS:341 */
                if (rep > 0) {
                    const int tgt = (g >= 0) ? g : (int)acnt[k] - 1;            /* reward[-1], TIS:346 */
                    if (tgt >= 0) q5[tgt] = 1; else PVE_ATOMIC_ADD(&misc[M_Q5U], 1);
                }
                del[k] = 1;                                                      /* TIS:348 */
                PVE_ATOMIC_ADD(&misc[M_NREM], 1);
                if (g >= 0) { status[g] = PVE_ST_DONE | PVE_ST_REMOVED; hdra[g] = -1; }   /* TIS:347-349 */
            } else if (p < 0 && (fl & PVE_F_CONTROL)) {                          /* TIS:350 */
                fl = (fl & ~(uint32_t)(PVE_F_CONTROL | PVE_F_LOCK)) | PVE_F_FINISH;      /* TIS:351-355 */
                status[g] = PVE_ST_DONE | PVE_ST_FINISHED;
                hdra[g] = -1;
                fin5[g] = 1;                                                     /* TIS:357 */
                PVE_ATOMIC_ADD(&misc[M_PASSED], 1);                              /* TIS:356 */
                PVE_ATOMIC_ADD(&misc[M_PSTEP], (int)(pk & 0xFFFFu));             /* TIS:359 */
            }
            const uint32_t c8 = fin > 255 ? 255u : (uint32_t)fin;
            spk[k] = (pk & 0xFFFFu) | (c8 << 16) | (fl << 24);
            fbits[k] = del[k] ? 0 : 1;                                           /* survivor flag */
            if (!del[k] && (fl & PVE_F_CONTROL)) PVE_ATOMIC_ADD(&misc[M_NCTRL], 1);
        }
    PVE_END_TID_NOSYNC

    /* ---- removal by stream compaction (TIS:435-444): survivors keep their order.  Every thread scans
     *      the survivor flags it wrote itself; the scan's barrier also publishes phase H ----------- */
    pve_block_excl_scan<NS, NT>(fbits, surv, V, wsum);
    PVE_FOR_TEAM(tid)
        (void)tid;
    PVE_END_TEAM

    /* ---- I: deadlock scan (TIS:365-370 + 1469-1499); final rewards; per-agent outputs ------ */
    PVE_FOR_TEAM(tid)
#ifndef __CUDACC__
        if (tid < PVE_NLANE) misc[M_NEXT0 + tid] = hdr->next_spawn[tid];        /* serial stand-in for J's ballot */
#endif
#pragma unroll 1
        for (int g = tid; g < A; g += NS) {
            const int k = vidx[g];
            /* reward[-1] overrides in processing order: a later -10 beats the agent's own +5 (Q5) */
            if (q5[g]) rew[g] = -10.f;                                           /* TIS:346 */
            else if (fin5[g]) rew[g] = 5.f;                                      /* TIS:357 */
            if (out_ok) {                                                        /* the small per-agent outputs */
                if (O.reward) O.reward[obase + g] = rew[g];
                if (O.ids) {
                    pve_v4 id; id.x = (uint32_t)b; id.y = lane_of[k];
                    id.z = (uint32_t)(k - lane_off[lane_of[k]]); id.w = (uint32_t)suid[k];
                    ((pve_v4 *)O.ids)[obase + g] = id;
                }
                if (O.cpv) O.cpv[obase + g] = cpv[g];
                if (O.status) O.status[obase + g] = status[g];
                if (O.jerk_sum) O.jerk_sum[obase + g] = (float)sjs[k];
                if (O.packed) {                                                  /* pve_agent_record */
                    const uint32_t c8 = cpv[g] > 255 ? 255u : (uint32_t)cpv[g];
                    pve_v4 rec;
                    rec.x = pve_fbits(rew[g]); rec.y = (uint32_t)suid[k];
                    rec.z = (uint32_t)lane_of[k] | ((uint32_t)(k - lane_off[lane_of[k]]) << 8) | ((uint32_t)status[g] << 16) | (c8 << 24);
                    rec.w = pve_fbits((float)sjs[k]);
                    ((pve_v4 *)O.packed)[obase + g] = rec;
                }
            }
            inct[g] = 0;                                                         /* from here on: ring length, set for the ring's reporter */
            if (!((spk[k] >> 24) & PVE_F_CONTROL) || del[k]) continue;
            int t = g, len = 0;
#pragma unroll 1
            for (int hop = 1; hop <= 10; ++hop) {                                /* TIS:1470-1478 */
                t = (t >= 0 && len == 0) ? (int)hdra[t] : -1;
                len = (t == g) ? hop : len;
            }
            if (len == 0) continue;
            slock[k] = 1;                                                        /* TIS:1482 */
            /* record_.sort() (TIS:1492) orders the ring's [vir_dis, follower, header] records; follower ids are
             * unique, so (vir_dis, follower agent index) is the whole key.  Every member of the ring walks it once and
             * finds its own rank and the ring's first member in (lane, j) order, mn (the reporter: TIS:365-370 calls
             * check_lock for it first); then it deposits its vir_dis where the reporter, walking the ring from itself,
             * meets the values in sorted order: at the member `rank` hops after mn. */
            const double dg = vdis[g];
            int mn = g, hmn = 0, rank = 0;
            t = g;
#pragma unroll 1
            for (int hop = 1; hop < len; ++hop) {
                t = hdra[t];
                const double dd = vdis[t];
                rank += (dd < dg || (dd == dg && t < g)) ? 1 : 0;
                if (t < mn) { mn = t; hmn = hop; }
            }
            int tgt = hmn + rank;
            tgt = tgt >= len ? tgt - len : tgt;
            t = g;
#pragma unroll 1
            for (int hop = 0; hop < tgt; ++hop) t = hdra[t];
            rsort[t] = dg;
            if (rank == 0) nn0[mn] = (uint16_t)g;                                /* record_[0]'s follower */
            if (mn == g) { inct[g] = len; PVE_ATOMIC_ADD(&misc[M_LOCK], 1); }
        }
    PVE_END_TEAM

    /* ---- J: arrivals (TIS:378-433) and header, one lane of warp 0 per traffic lane -------------- */
    PVE_FOR_TEAM(tid)
        /* the reporter of every ring: sum(dis) over the sorted records and the unlock rule, TIS:1495-1497 */
#pragma unroll 1
        for (int g = tid; g < A; g += NS) {
            const int len = inct[g];
            if (len == 0) continue;
            double sum = 0;
            int t = g;
#pragma unroll 1
            for (int hop = 0; hop < len; ++hop) { sum = sum + rsort[t]; t = hdra[t]; }
            if (rsort[g] < P.thr || sum / (double)len < P.thr + 3) {             /* TIS:1495 */
                const int first_o = nn0[g];
                slocka[vidx[first_o]] = 1;                                       /* TIS:1496 */
                slocka[vidx[hdra[first_o]]] = -1;                                /* TIS:1497 */
            }
        }
        if (tid < 32) {
            const int i = tid < PVE_NLANE ? tid : 0;
            const int tick = hdr->tick + 1;                                      /* TIS:223 */
            const int total = surv[V], nctrl = misc[M_NCTRL];
            int room = VC - total;
            room = (AC - nctrl) < room ? (AC - nctrl) : room;
            const int surv_i = (int)surv[lane_off[i + 1]] - (int)surv[lane_off[i]];
            const int want = (tid < PVE_NLANE && tick >= hdr->next_spawn[i] && surv_i < 255) ? 1 : 0;   /* TIS:379 */
            /* arrivals are granted in lane order while there is room (capacity is a sticky error) */
#ifdef __CUDACC__
            const unsigned wants = __ballot_sync(0xffffffffu, want);
            const int before = __popc(wants & ((1u << tid) - 1u));
            const int n_want = __popc(wants);
#else
            int before = 0, n_want = 0;
            for (int q2 = 0; q2 < PVE_NLANE; ++q2) {
                const int sq = (int)surv[lane_off[q2 + 1]] - (int)surv[lane_off[q2]];
                const int wq = (tick >= misc[M_NEXT0 + q2] && sq < 255) ? 1 : 0;
                if (q2 < i) before += wq;
                n_want += wq;
            }
#endif
            if (tid < PVE_NLANE) {
                const int sp_i = (want && before < room) ? 1 : 0;
                const int pref = before < room ? before : (room > 0 ? room : 0);
                misc[M_SPAWN0 + i] = sp_i;
                misc[M_SPREF0 + i] = pref;
                if (want && !sp_i) PVE_ATOMIC_ADD(&hdr->overflow, 1);
                /* head of the rebuilt virtual lane, read by next tick's step() (Q2) */
                if (hdr->lane_n[i] > 0) {
                    const int kh = headk[i];
                    if (kh >= 0) {
                        hdr->head_lane[i] = (int8_t)lane_of[kh];
                        hdr->head_j[i] = (uint8_t)(kh - lane_off[lane_of[kh]]);
                    } else { hdr->head_lane[i] = -1; hdr->head_j[i] = 0; }
                }
                if (sp_i) {
                    const int rec = (int)hdr->veh_rec[i] + 1;                    /* TIS:430 */
                    hdr->veh_rec[i] = (uint16_t)rec;
                    if constexpr (POI) {
                        const size_t q = (size_t)b * PVE_NLANE + i;
                        hdr->next_spawn[i] = pve_next_arrival(arr, b, i, rec, arr.pend + q, arr.mean[q]);
                    } else {
                        hdr->next_spawn[i] = (rec < P.K) ? arr[((size_t)b * P.K + rec) * PVE_NLANE + i] : PVE_NEVER;
                    }
                }
                hdr->lane_n[i] = (uint8_t)(surv_i + sp_i);
                if (i == PVE_NLANE - 1) {            /* last in serial order: nobody reads hdr->tick after it */
                    const int granted = n_want < room ? n_want : (room > 0 ? room : 0);
                    misc[M_SPREF0 + PVE_NLANE] = granted;
                    hdr->n_veh = total + granted;
                    hdr->n_ctrl = nctrl + granted;
                    misc[M_IDSEQ0] = hdr->id_seq;
                    hdr->id_seq += granted;                                      /* TIS:433 */
                    hdr->tick = tick;
                    hdr->passed_veh += misc[M_PASSED];
                    hdr->passed_step_total += misc[M_PSTEP];
                    if (!out_ok) PVE_ATOMIC_ADD(&hdr->overflow, 1);              /* output rows do not fit */
                }
            }
        }
    PVE_END_TEAM

    /* ---- K: write the state back, compacted; header; statistics ---------------------------------- */
    pve_warp0_sums<NT>(rew, fin5, sjs, vidx, A, dsum);
    PVE_FOR_TEAM(tid)
#pragma unroll 1
        for (int k = tid; k < V; k += NS)
            if (!del[k]) {
                const size_t o = vbase + (size_t)((int)surv[k] + misc[M_SPREF0 + lane_of[k]]);
                S.p[o] = sp[k]; S.v[o] = sv[k]; S.a[o] = sa[k]; S.js[o] = sjs[k];
                pve_veh_meta mt;
                mt.uid = suid[k];
                mt.packed = spk[k] | ((uint32_t)(slock[k] ? PVE_F_LOCK : 0) << 24)
                            | ((uint32_t)(slocka[k] + 1) << 27);
                S.meta[o] = mt;
            }
        if (tid < PVE_NLANE && misc[M_SPAWN0 + tid]) {                           /* TIS:395-427 */
            const int i = tid;
            const int np = (int)surv[lane_off[i + 1]] + misc[M_SPREF0 + i];
            const size_t o = vbase + (size_t)np;
            S.p[o] = P.spawn_p[i % 3]; S.v[o] = P.v0; S.a[o] = 0.0; S.js[o] = 0.0;
            pve_veh_meta mt;
            mt.uid = misc[M_IDSEQ0] + misc[M_SPREF0 + i];
            mt.packed = ((uint32_t)PVE_F_CONTROL << 24) | (1u << 27);
            S.meta[o] = mt;
            pve_v4 z; z.x = 0; z.y = 0; z.z = 0; z.w = 0;
            for (int q = 0; q < PVE_OBS_W / 4; ++q) ((pve_v4 *)(row0_next + (size_t)np * PVE_OBS_W))[q] = z;
        }
        /* stored row 0 of every surviving agent -> next tick's neighbour rows / actor input */
#pragma unroll 1
        for (int it = tid; it < A * 8; it += NS) {
            const int g = it >> 3, q = it & 7;
            const int k = vidx[g];
            if (q < 7 && !del[k]) {
                const int np = (int)surv[k] + misc[M_SPREF0 + lane_of[k]];
                ((pve_v4 *)(row0_next + (size_t)np * PVE_OBS_W))[q] = ((const pve_v4 *)(row0 + (size_t)g * PVE_OBS_W))[q];
            }
        }
        if (tid >= 32 && tid < 32 + PVE_HDR_BYTES / 16) ((pve_v4 *)(S.hdr + b))[tid - 32] = ((const pve_v4 *)hdr)[tid - 32];
        /* the scalar tail of the tick on two different warps: the last team thread publishes the counts, the class
         * of the next tick and the per-intersection outputs; lanes 0-9 of warp 0 add one statistic each */
        if (tid == NS - 1) {
            S.n_ctrl_next[b] = hdr->n_ctrl; S.n_veh[b] = hdr->n_veh;
            PVE_RED_ADD(&S.gs_acc[b >> PVE_GROUP_SHIFT], hdr->n_ctrl);         /* next tick's group sums */
            if ((b & ((1 << PVE_GROUP_SHIFT) - 1)) == 0) S.gs_zero[b >> PVE_GROUP_SHIFT] = 0;
            if (S.klass_next) {      /* next tick: vehicles stepped + arrivals already due must fit the small class */
                int due = 0;
#pragma unroll
                for (int i = 0; i < PVE_NLANE; ++i) due += (hdr->tick + 1 >= hdr->next_spawn[i]) ? 1 : 0;
                const int big = (hdr->n_veh + due > S.small_vc || hdr->n_ctrl + due > S.small_ac) ? 1 : 0;
                S.klass_next[b] = (uint8_t)big;
                if (big) S.big_list_next[PVE_ATOMIC_ADD(S.big_cnt_next, 1)] = b;
                if (b == 0) *S.big_cnt_zero = 0;
            }
            if (O.agent_offset) {
                O.agent_offset[b] = (int32_t)obase;
                if (b == P.B - 1) O.agent_offset[P.B] = (int32_t)obase + A;
            }
            if (O.env_collisions) O.env_collisions[b] = misc[M_COLL];
            if (O.env_lock) O.env_lock[b] = misc[M_LOCK];
            if (O.env_removed) O.env_removed[b] = misc[M_NREM];
        }
        if (tid < PVE_NSTAT) {
            /* per-intersection running statistics (end-of-rollout reduction, MAIN:407-415); dsum: pve_warp0_sums */
            static_assert(PVE_STAT_AGENT == 0 && PVE_STAT_VEH == 1 && PVE_STAT_COLL == 2 && PVE_STAT_LOCK == 3 && PVE_STAT_JERK == 4 &&
                          PVE_STAT_RSUM == 5 && PVE_STAT_RSQ == 6 && PVE_STAT_REMOVED == 7 && PVE_STAT_STEPS == 8 && PVE_STAT_Q5U == 9,
                          "statistic order");
            const int iv = tid == 0 ? A : tid == 1 ? V : tid == 2 ? misc[M_COLLAG] : tid == 3 ? misc[M_LOCK]
                         : tid == 7 ? misc[M_NREM] : tid == 8 ? 1 : misc[M_Q5U];
            const double val = tid == 4 ? dsum[2] : tid == 5 ? dsum[0] : tid == 6 ? dsum[1] : (double)iv;
            PVE_RED_ADD(&S.stats[(size_t)b * PVE_NSTAT + tid], val);
        }
    PVE_END_TID_NOSYNC

    /* ---- optional output: where the 7 observation rows of every agent were copied from (pve_outputs.nbr_src).
     *      Only in the SRC instantiation of the kernel. */
    if (SRC && O.nbr_src != nullptr && out_ok) {
        PVE_FOR_TEAM(tid)
#pragma unroll 1
            for (int g = tid; g < A; g += NS) {
                uint32_t w4[4];
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const uint32_t c = q < PVE_OBS_H ? srcc[g * 7 + q] : (uint32_t)(AC * 7);
                    const uint32_t v = c == (uint32_t)(AC * 7) ? 0xFFFFu
                                       : (c & PVE_SRC_PREV) ? (0x4000u | ((c & 0x7FFFu) / 7u)) : c / 7u;
                    if (q & 1) w4[q >> 1] |= v << 16; else w4[q >> 1] = v;
                }
                pve_v4 nb; nb.x = w4[0]; nb.y = w4[1]; nb.z = w4[2]; nb.w = w4[3];
                ((pve_v4 *)O.nbr_src)[obase + g] = nb;
            }
        PVE_END_TID_NOSYNC
    }
    /* ---- optional output: the factored observation, on the half of the CTA that has no observation rows to move (the
     *      mover warps took it after G1 when pve_outputs.obs is null) */
    if (SRC && (NS == NT || oblk != nullptr)) {
        PVE_FOR_TEAM(tid)
            pve_write_factored(FJ, tid, NS);
        PVE_END_TID_NOSYNC
    }

    /* ---- N: observation rows leave the SM (already under way on the upper half when the CTA is split) */
#ifdef __CUDACC__
    if (NS == NT) pve_move_rows<NT, NT / 32>(RJ, 0);
#else
    pve_move_rows<NT, 1>(RJ, 0);
#endif
#if defined(PVE_PHASE_TIMING) && defined(__CUDACC__)
    if (threadIdx.x == 0 && S.stats) {      /* debug build: overwrite this intersection's stats rows with stamps */
        long long *dbg = (long long *)S.dbg + (size_t)b * 48;
        for (int q = 0; q < 40; ++q) dbg[q] = q < pve_nstamp ? pve_stamp[q] - pve_stamp[0] : -1;
        unsigned long long gt1; unsigned smid;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt1));
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        dbg[40] = pve_stamp[0]; dbg[41] = (long long)pve_gt0; dbg[42] = (long long)gt1; dbg[43] = smid;
        dbg[44] = A; dbg[45] = V;                            /* dbg[47]: the row movers' last clock */
    }
#endif
}
