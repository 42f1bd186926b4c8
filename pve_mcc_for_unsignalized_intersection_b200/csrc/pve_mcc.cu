/*
 * pve_mcc.cu -- C ABI (include/pve_mcc.h) and kernel launches of the batched PVE-MCC
 * environment step for B200 (sm_100a).
 *
 * Build (see __graft_entry__.build):
 *   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -fmad=false -shared
 *        -Xcompiler -fPIC -I include pve_mcc.cu -o libpve_mcc.so
 *
 * With -DPVE_HOST_EMULATION and g++ the same file builds the sequential kernel-logic
 * emulation used ONLY by the CPU test tier (tests/emul/); pve_backend() tells them apart and
 * the Python product wrapper refuses anything but the CUDA backend.
 */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <new>

#include "scene_step.cuh"
#include "scene_step4.cuh"
#include "actor_mma.cuh"
#include "nstep.cuh"
#include "critic_mma.cuh"
#include "mlp_tc5.cuh"

#ifndef PVE_HOST_EMULATION
#include <cuda_runtime.h>
#define PVE_BACKEND "cuda-sm_100a"
typedef cudaStream_t pve_stream_t;
#else
#define PVE_BACKEND "host-emulation(test-only)"
typedef void *pve_stream_t;
#endif

namespace {

const int8_t kLane2Lane[PVE_NLANE][4] = {            /* TIS:153-166 */
    {10, 3, 9, 7}, {10, 6, 3, 4}, {-1, -1, -1, -1}, {1, 6, 0, 10}, {1, 9, 6, 7}, {-1, -1, -1, -1},
    {4, 9, 3, 1},  {4, 0, 9, 10}, {-1, -1, -1, -1}, {7, 0, 6, 4},  {7, 3, 0, 1}, {-1, -1, -1, -1}};

}  // namespace

#define PVE_ASYNC_SLOTS 3      /* ticks in flight on the pipelined host path */

struct pve_scene {
    pve_config cfg;
    PveParams prm;
    PveState st;
    int device;
    int threads;
    size_t smem_bytes;
    int phase;
    int rot;                     /* which of the three group-sum buffers holds this tick's counts */
    int32_t *gsum;               /* [3][G] */
    int n_groups;
    int32_t *n_ctrl_buf[2];      /* ping-pong with `phase` */
    int32_t *order;              /* busiest-first CTA order */
    /* lane_num = 4 (row N3): its own kernel, one warp per intersection; dense output offsets from a scan kernel */
    int lane_num;
    Pve4Params prm4;
    const uint8_t *draws;        /* lane_num = 8: intention draws [B][K][12] (borrowed, pve_set_intention_draws) */
    int64_t *off4;               /* [B + 1] */
    /* dual mode (default class, default CTA size): two concurrent kernels per tick, see PveState::klass */
    int dual, dual_pdl;
    uint8_t *klass_buf[2];       /* ping-pong with `phase` */
    int32_t *big_list_buf[2];
    int32_t *big_cnt3;           /* [3], rotates with `rot` */
#ifndef PVE_HOST_EMULATION
    cudaStream_t side;           /* the big kernel's stream */
    cudaEvent_t ev_fork, ev_join;
    /* pipelined host path (pve_step_host_async): copy-in / copy-out streams, two ticks in flight */
    cudaStream_t s_in, s_out, s_cnt;
    cudaEvent_t a_in[PVE_ASYNC_SLOTS], a_k[PVE_ASYNC_SLOTS], a_cnt[PVE_ASYNC_SLOTS], a_done[PVE_ASYNC_SLOTS];
    float *a_act[PVE_ASYNC_SLOTS];       /* device action buffers */
    int64_t *a_total;                    /* pinned [PVE_ASYNC_SLOTS]: rows of the tick AFTER the one in the slot */
    int64_t a_rows[PVE_ASYNC_SLOTS];
    int64_t a_seq, a_waited;             /* ticks enqueued / waited for; slot = tick % PVE_ASYNC_SLOTS */
    int a_ready;                         /* streams/events created */
    int64_t a_copied;                    /* ticks whose copy-out has been enqueued */
    pve_outputs a_odev[PVE_ASYNC_SLOTS], a_ohost[PVE_ASYNC_SLOTS];
    int32_t a_mask[PVE_ASYNC_SLOTS];
#endif
    int order_age;               /* ticks since the order was refreshed (-1: never) */
    const int32_t *spawn_tick;   /* borrowed */
    /* Poisson mode (pve_reset_poisson / _rates): the step kernels generate the arrivals (arrivals.cuh) instead of
     * reading spawn_tick; pend_dev / clock_dev are allocated by the first Poisson reset and kept for the handle's
     * lifetime */
    int poisson;
    PvePoisson poi;
    double *pend_dev;            /* [2][B][12]: PvePoisson::pend, then PvePoisson::mean */
    double *clock_dev;           /* [PVE_MAX_TICK + 1] */
    float *actions_dev;          /* staging for pve_step_host */
    double *counters_dev;
    int32_t *pinned_i32;         /* host-visible scratch */
    int32_t *pinned_gs;          /* host copy of the group sums (next agent total) */
    int64_t next_total;          /* rows of the next tick if known, else -1 */
    int profiling;               /* record events around the step and scan kernels */
    size_t smem_pad;             /* experiment knob (env PVE_SMEM_PAD): extra dynamic shared memory per CTA */
    int exp_no_obs;
    int host_zerocopy;           /* pve_step_host reads/writes pinned host buffers in place (env PVE_HOST_ZEROCOPY=0: staged copies) */
#ifndef PVE_HOST_EMULATION
    cudaEvent_t ev[3];
#endif
    char err[512];
};

/* =============================================================================================
 * runtime layer: CUDA, or plain host memory for the test-only emulation
 * =========================================================================================== */
#ifndef PVE_HOST_EMULATION
#define RT_CHECK(s, call)                                                                     \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess) {                                                              \
            snprintf((s)->err, sizeof((s)->err), "%s failed: %s (%s:%d)", #call,              \
                     cudaGetErrorString(e_), __FILE__, __LINE__);                             \
            return PVE_ECUDA;                                                                 \
        }                                                                                     \
    } while (0)
static cudaError_t rt_alloc(void **p, size_t n) { return cudaMalloc(p, n ? n : 16); }
static void rt_free(void *p) { if (p) cudaFree(p); }
static cudaError_t rt_memset(void *p, int v, size_t n, pve_stream_t s) { return cudaMemsetAsync(p, v, n, s); }
static cudaError_t rt_copy(void *d, const void *s, size_t n, pve_stream_t st) {
    return cudaMemcpyAsync(d, s, n, cudaMemcpyDefault, st);
}
static cudaError_t rt_sync(pve_stream_t s) { return cudaStreamSynchronize(s); }
static cudaError_t rt_host_alloc(void **p, size_t n) { return cudaHostAlloc(p, n, cudaHostAllocDefault); }
static void rt_host_free(void *p) { if (p) cudaFreeHost(p); }
#else
#define RT_CHECK(s, call)                                                                     \
    do {                                                                                      \
        if ((call) != 0) {                                                                    \
            snprintf((s)->err, sizeof((s)->err), "%s failed (%s:%d)", #call, __FILE__, __LINE__); \
            return PVE_ECUDA;                                                                 \
        }                                                                                     \
    } while (0)
static int rt_alloc(void **p, size_t n) { *p = calloc(1, n ? n : 16); return *p ? 0 : 1; }
static void rt_free(void *p) { free(p); }
static int rt_memset(void *p, int v, size_t n, pve_stream_t) { memset(p, v, n); return 0; }
static int rt_copy(void *d, const void *s, size_t n, pve_stream_t) { memmove(d, s, n); return 0; }
static int rt_sync(pve_stream_t) { return 0; }
static int rt_host_alloc(void **p, size_t n) { return rt_alloc(p, n); }
static void rt_host_free(void *p) { free(p); }
#endif

/* =============================================================================================
 * kernels
 * =========================================================================================== */
#ifndef PVE_HOST_EMULATION

/* register budget: as many CTAs per SM as the class's shared memory admits (8 for 128/80, 7 for
 * 128/96), counted in 128-thread units */
#ifndef PVE_MAX_RESIDENT
#define PVE_MAX_RESIDENT 8     /* experiment knob: cap on the CTAs per SM the register budget is sized for */
#endif
template <int VC, int AC>
struct PveResident {
    static constexpr int BY_SMEM = 233472 / (int)(PveLayout<VC, AC>::BYTES + 1024);
    static constexpr int CTAS128 = BY_SMEM < PVE_MAX_RESIDENT ? BY_SMEM : PVE_MAX_RESIDENT;     /* in 128-thread units */
    /* 96-thread CTAs (3 warps): as many as shared memory admits, which leaves up to 85 registers per thread */
    /* 512-thread CTAs (large classes): two per SM when shared memory admits them, i.e. a 64-register budget */
    static constexpr int blocks(int nt) {
        return nt == 96 ? BY_SMEM : nt == 512 ? (BY_SMEM < 2 ? BY_SMEM : 2) : (CTAS128 * 128 / nt > 0 ? CTAS128 * 128 / nt : 1);
    }
};
template <int NT, int VC, int AC, bool SRC, bool POI>
__global__ void __launch_bounds__(NT, PveResident<VC, AC>::blocks(NT))
pve_step_kernel(const PveParams P, const PveState S, const pve_outputs O, const typename PveArrivalsT<POI>::type spawn_tick,
                const float *actions, const int phase) {
    extern __shared__ __align__(16) unsigned char pve_smem[];
    /* CTAs are dispatched in index order; starting the busiest intersections first shortens the tail
     * of the launch (a CTA lives ~22 us, a launch of 4096 ~100 us) */
    const int b = S.order ? S.order[blockIdx.x] : (int)blockIdx.x;
    /* dual mode: intersections of the big kernel are skipped (pve_step_block tests klass[b] after it has issued its
     * first loads, so the test costs no extra memory round trip) */
    pve_step_block<NT, VC, AC, SRC, POI>(P, S, O, spawn_tick, actions, phase, b, pve_smem, S.klass);
    /* dual mode launches this grid as the programmatic dependent of the big kernel (same stream, started while the
     * big kernel runs): it may not complete before that one has (no-op for an ordinary launch) */
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

/* dual mode: the intersections that do not fit the small class, a few per tick */
template <int NT, int VC, int AC, bool SRC, bool POI>
__global__ void __launch_bounds__(NT, PveResident<VC, AC>::blocks(NT))
pve_step_big_kernel(const PveParams P, const PveState S, const pve_outputs O, const typename PveArrivalsT<POI>::type spawn_tick,
                    const float *actions, const int phase) {
    extern __shared__ __align__(16) unsigned char pve_smem[];
    asm volatile("griddepcontrol.launch_dependents;");      /* the small kernel shares nothing with this one: start it now */
    const int n = *S.big_cnt;
    for (int i = (int)blockIdx.x; i < n; i += (int)gridDim.x) {
        pve_step_block<NT, VC, AC, SRC, POI>(P, S, O, spawn_tick, actions, phase, S.big_list[i], pve_smem, nullptr);
        __syncthreads();                                   /* shared memory is reused by the next one */
    }
}

/* pipelined host path: next tick's row count, written straight into (mapped) pinned host memory -- a DMA copy for
 * these few bytes would queue behind the bulk copies of the copy engines */
__global__ void pve_total_kernel(const int32_t *__restrict__ gs, int G, volatile int64_t *total_host) {
    int64_t t = 0;
    for (int g = threadIdx.x; g < G; g += 32) t += gs[g];
    for (int d = 16; d > 0; d >>= 1) t += __shfl_xor_sync(0xffffffffu, t, d);
    if (threadIdx.x == 0) *total_host = t;
}

/* dual mode, after reset / set_state: classes and the big kernel's list from the headers */
__global__ void pve_classify_kernel(PveState S, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const pve_env_header *h = S.hdr + b;
    int due = 0;
    for (int i = 0; i < PVE_NLANE; ++i) due += (h->tick + 1 >= h->next_spawn[i]) ? 1 : 0;
    const int big = (h->n_veh + due > S.small_vc || h->n_ctrl + due > S.small_ac) ? 1 : 0;
    S.klass_next[b] = (uint8_t)big;
    if (big) S.big_list_next[atomicAdd(S.big_cnt_next, 1)] = b;
}

/* ---- lane_num = 4 / 8 (scene_step4.cuh): one warp per intersection, PVE4_WARPS intersections per CTA -------------- */
#define PVE4_WARPS 4
template <int NLN, int LC, bool POI, bool SRC>
__global__ void __launch_bounds__(32 * PVE4_WARPS)
pve4_step_kernel(const Pve4Params P, const PveState S, const pve_outputs O, const typename PveArrivalsT<POI>::type spawn_tick,
                 const uint8_t *draws, const float *actions, const int64_t *off4) {
    extern __shared__ __align__(16) unsigned char pve_smem[];
    const int b = (int)blockIdx.x * PVE4_WARPS + (int)(threadIdx.x >> 5);
    if (b >= P.B) return;
    Pve4SmemT<LC> &M = ((Pve4SmemT<LC> *)pve_smem)[threadIdx.x >> 5];
    pve4_step_block<NLN, POI, SRC>(P, S, O, spawn_tick, draws, actions, b, M, off4[b]);
}

/* exclusive prefix of the agent counts -> first output row of every intersection (one CTA; B is small on this path) */
__global__ void __launch_bounds__(1024)
pve4_offsets_kernel(const int32_t *__restrict__ n_ctrl, int64_t *__restrict__ off, int B) {
    __shared__ int64_t part[1024];
    const int tid = threadIdx.x, per = (B + 1023) / 1024;
    const int lo = tid * per, hi = min(B, lo + per);
    int64_t s = 0;
    for (int b = lo; b < hi; ++b) s += n_ctrl[b];
    part[tid] = s;
    __syncthreads();
    if (tid == 0) { int64_t run = 0; for (int t = 0; t < 1024; ++t) { const int64_t c = part[t]; part[t] = run; run += c; } off[B] = run; }
    __syncthreads();
    int64_t run = part[tid];
    for (int b = lo; b < hi; ++b) { off[b] = run; run += n_ctrl[b]; }
}

/* order[i] = intersections sorted by their agent count, descending (counting sort, one CTA) */
__global__ void __launch_bounds__(1024)
pve_order_kernel(const int32_t *__restrict__ n_ctrl, int32_t *__restrict__ order, int B) {
    __shared__ int hist[1025];
    const int tid = threadIdx.x;
    for (int i = tid; i < 1025; i += 1024) hist[i] = 0;
    __syncthreads();
    for (int b = tid; b < B; b += 1024) atomicAdd(&hist[1023 - min(max(n_ctrl[b], 0), 1023)], 1);
    __syncthreads();
    if (tid == 0) {
        int run = 0;
        for (int i = 0; i < 1024; ++i) { const int c = hist[i]; hist[i] = run; run += c; }
    }
    __syncthreads();
    for (int b = tid; b < B; b += 1024) order[atomicAdd(&hist[1023 - min(max(n_ctrl[b], 0), 1023)], 1)] = b;
}

/* group sums of n_ctrl after reset / set_state (during a rollout the step kernel maintains them) */
__global__ void pve_gsum_kernel(const int32_t *__restrict__ n_ctrl, int32_t *__restrict__ gs_now,
                                int32_t *__restrict__ gs_a, int32_t *__restrict__ gs_b, int B, int G) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    int s = 0;
    for (int i = g << PVE_GROUP_SHIFT; i < min(B, (g + 1) << PVE_GROUP_SHIFT); ++i) s += n_ctrl[i];
    gs_now[g] = s; gs_a[g] = 0; gs_b[g] = 0;
}

template <bool POI>
__global__ void pve_reset_kernel(PveState S, const typename PveArrivalsT<POI>::type spawn_tick, int B, int K, int warmup) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    pve_env_header h;
    memset(&h, 0, sizeof h);
    int first = PVE_NEVER;
    for (int i = 0; i < PVE_NLANE; ++i) {
        int t;
        if constexpr (POI) t = pve_reset_lane(spawn_tick, b, i);
        else t = (K > 0) ? spawn_tick[(size_t)b * K * PVE_NLANE + i] : PVE_NEVER;
        h.next_spawn[i] = t;
        h.head_lane[i] = -1;
        first = min(first, t);
    }
    /* TIS:214-220: empty scene updates until the first arrival; the tick that spawns it is run by
     * pve_reset as an ordinary (empty) step */
    h.tick = (warmup && first != PVE_NEVER) ? max(first - 1, 0) : 0;
    S.hdr[b] = h;
    S.n_ctrl[b] = 0;
    S.n_veh[b] = 0;
    for (int q = 0; q < PVE_NSTAT; ++q) S.stats[(size_t)b * PVE_NSTAT + q] = 0.0;
}

/* after pve_set_state: recompute the derived header fields */
template <bool POI>
__global__ void pve_recount_kernel(PveState S, const typename PveArrivalsT<POI>::type spawn_tick, int B, int VC, int K) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    pve_env_header *h = S.hdr + b;
    int nv = 0, nc = 0;
    for (int i = 0; i < PVE_NLANE; ++i) nv += h->lane_n[i];
    nv = min(nv, VC);
    for (int k = 0; k < nv; ++k) nc += (S.meta[(size_t)b * VC + k].packed >> 24) & PVE_F_CONTROL;
    h->n_veh = nv;
    h->n_ctrl = nc;
    for (int i = 0; i < PVE_NLANE; ++i) {
        const int rec = h->veh_rec[i];
        if constexpr (POI) h->next_spawn[i] = pve_recount_lane(spawn_tick, b, i, rec);
        else h->next_spawn[i] = (spawn_tick && rec < K) ? spawn_tick[((size_t)b * K + rec) * PVE_NLANE + i] : PVE_NEVER;
    }
    S.n_ctrl[b] = nc;
    S.n_veh[b] = nv;
}

/* K5: end-of-rollout statistics, one CTA, deterministic order */
__global__ void __launch_bounds__(256)
pve_stats_kernel(PveState S, int B, double *out) {
    __shared__ double sh[16][256];
    const int tid = threadIdx.x;
    double acc[16];
    for (int q = 0; q < 16; ++q) acc[q] = 0;
    for (int b = tid; b < B; b += 256) {
        const double *st = S.stats + (size_t)b * PVE_NSTAT;
        const pve_env_header *h = S.hdr + b;
        acc[0] += st[PVE_STAT_AGENT]; acc[1] += st[PVE_STAT_VEH];
        acc[2] += st[PVE_STAT_STEPS]; acc[13] += st[PVE_STAT_Q5U];
        acc[3] += (double)h->id_seq; acc[4] += (double)h->passed_veh; acc[5] += (double)h->passed_step_total;
        acc[6] += st[PVE_STAT_JERK]; acc[7] += st[PVE_STAT_COLL]; acc[8] += st[PVE_STAT_LOCK];
        acc[9] += st[PVE_STAT_RSUM]; acc[10] += st[PVE_STAT_RSQ]; acc[11] += st[PVE_STAT_REMOVED];
        acc[12] += (double)h->overflow;
    }
    for (int q = 0; q < 16; ++q) sh[q][tid] = acc[q];
    __syncthreads();
    if (tid < 16) {
        double s = 0;
        for (int t = 0; t < 256; ++t) s += sh[tid][t];
        out[tid] = s;
    }
}

/* pve_expand_obs: one CTA per intersection; consecutive threads store consecutive 16-byte pieces of its block (the
 * code of a row is read by the 7 threads of its pieces) */
__global__ void __launch_bounds__(128)
pve_expand_obs_kernel(const int32_t *__restrict__ off, int64_t out_cap, const pve_v4 *__restrict__ r0,
                      const pve_v4 *__restrict__ pr, const int16_t *__restrict__ src, pve_v4 *__restrict__ obs) {
    const int b = (int)blockIdx.x;
    const int64_t o0 = off[b], o1 = off[b + 1];
    if (o0 < 0 || o1 < o0 || o1 > out_cap) return;           /* rows the step did not write (out_cap) */
    const int64_t n = (o1 - o0) * (PVE_OBS_H * 7);
    for (int64_t it = threadIdx.x; it < n; it += blockDim.x) {
        const int64_t g = it / (PVE_OBS_H * 7);
        const int rem = (int)(it - g * (PVE_OBS_H * 7)), q = rem / 7, piece = rem - q * 7;
        int64_t idx = 0;
        const int k = pve_obs_src_decode(src[(o0 + g) * 8 + q], o1 - o0, &idx);
        pve_v4 v;
        if (k > 0) v = (k == 1 ? r0 : pr)[(o0 + idx) * 7 + piece];
        else { const uint32_t w = k == 0 ? 0u : PVE_NAN_BITS; v.x = w; v.y = w; v.z = w; v.w = w; }
        obs[(o0 + g) * (PVE_OBS_H * 7) + rem] = v;
    }
}

#else  /* ------------------------------- host emulation ------------------------------------ */

static void emul_gsum(const int32_t *n_ctrl, int32_t *gs_now, int32_t *gs_a, int32_t *gs_b, int B, int G) {
    for (int g = 0; g < G; ++g) {
        int s = 0;
        for (int i = g << PVE_GROUP_SHIFT; i < B && i < ((g + 1) << PVE_GROUP_SHIFT); ++i) s += n_ctrl[i];
        gs_now[g] = s; gs_a[g] = 0; gs_b[g] = 0;
    }
}
template <bool POI>
static void emul_reset(PveState S, const typename PveArrivalsT<POI>::type spawn_tick, int B, int K, int warmup) {
    for (int b = 0; b < B; ++b) {
        pve_env_header h;
        memset(&h, 0, sizeof h);
        int first = PVE_NEVER;
        for (int i = 0; i < PVE_NLANE; ++i) {
            int t;
            if constexpr (POI) t = pve_reset_lane(spawn_tick, b, i);
            else t = (K > 0) ? spawn_tick[(size_t)b * K * PVE_NLANE + i] : PVE_NEVER;
            h.next_spawn[i] = t; h.head_lane[i] = -1;
            first = t < first ? t : first;
        }
        h.tick = (warmup && first != PVE_NEVER) ? (first - 1 > 0 ? first - 1 : 0) : 0;
        S.hdr[b] = h; S.n_ctrl[b] = 0; S.n_veh[b] = 0;
        for (int q = 0; q < PVE_NSTAT; ++q) S.stats[(size_t)b * PVE_NSTAT + q] = 0.0;
    }
}
template <bool POI>
static void emul_recount(PveState S, const typename PveArrivalsT<POI>::type spawn_tick, int B, int VC, int K) {
    for (int b = 0; b < B; ++b) {
        pve_env_header *h = S.hdr + b;
        int nv = 0, nc = 0;
        for (int i = 0; i < PVE_NLANE; ++i) nv += h->lane_n[i];
        nv = nv < VC ? nv : VC;
        for (int k = 0; k < nv; ++k) nc += (S.meta[(size_t)b * VC + k].packed >> 24) & PVE_F_CONTROL;
        h->n_veh = nv; h->n_ctrl = nc;
        for (int i = 0; i < PVE_NLANE; ++i) {
            const int rec = h->veh_rec[i];
            if constexpr (POI) h->next_spawn[i] = pve_recount_lane(spawn_tick, b, i, rec);
            else h->next_spawn[i] = (spawn_tick && rec < K) ? spawn_tick[((size_t)b * K + rec) * PVE_NLANE + i] : PVE_NEVER;
        }
        S.n_ctrl[b] = nc; S.n_veh[b] = nv;
    }
}
static void emul_stats(PveState S, int B, double *out) {
    for (int q = 0; q < 16; ++q) out[q] = 0;
    for (int b = 0; b < B; ++b) {
        const double *st = S.stats + (size_t)b * PVE_NSTAT;
        const pve_env_header *h = S.hdr + b;
        out[0] += st[PVE_STAT_AGENT]; out[1] += st[PVE_STAT_VEH];
        out[2] += st[PVE_STAT_STEPS]; out[13] += st[PVE_STAT_Q5U];
        out[3] += (double)h->id_seq; out[4] += (double)h->passed_veh; out[5] += (double)h->passed_step_total;
        out[6] += st[PVE_STAT_JERK]; out[7] += st[PVE_STAT_COLL]; out[8] += st[PVE_STAT_LOCK];
        out[9] += st[PVE_STAT_RSUM]; out[10] += st[PVE_STAT_RSQ]; out[11] += st[PVE_STAT_REMOVED];
        out[12] += (double)h->overflow;
    }
}
#endif

/* =============================================================================================
 * launch helpers
 * =========================================================================================== */
static void set_rotation(pve_scene *s) {
    const int G = s->n_groups;
    const int nc = s->lane_num == 12 ? s->phase : 0;      /* lane_num 4 / 8: one buffer, see launch_step4 */
    s->st.n_ctrl = s->n_ctrl_buf[nc];
    s->st.n_ctrl_next = s->n_ctrl_buf[nc ^ 1];
    s->st.gs_read = s->gsum + (size_t)(s->rot % 3) * G;
    s->st.gs_acc = s->gsum + (size_t)((s->rot + 1) % 3) * G;
    s->st.gs_zero = s->gsum + (size_t)((s->rot + 2) % 3) * G;
    if (s->dual) {
        s->st.klass = s->klass_buf[s->phase]; s->st.klass_next = s->klass_buf[s->phase ^ 1];
        s->st.big_list = s->big_list_buf[s->phase]; s->st.big_list_next = s->big_list_buf[s->phase ^ 1];
        s->st.big_cnt = s->big_cnt3 + s->rot % 3; s->st.big_cnt_next = s->big_cnt3 + (s->rot + 1) % 3;
        s->st.big_cnt_zero = s->big_cnt3 + (s->rot + 2) % 3;
    }
}

/* after reset / set_state: group sums from n_ctrl, rotation restarted */
static int32_t launch_gsum(pve_scene *s, pve_stream_t stream) {
    s->rot = 0;
    set_rotation(s);
    const int G = s->n_groups;
#ifndef PVE_HOST_EMULATION
    pve_gsum_kernel<<<(G + 127) / 128, 128, 0, stream>>>(s->st.n_ctrl, s->gsum, s->gsum + G, s->gsum + 2 * (size_t)G,
                                                          s->cfg.n_envs, G);
    RT_CHECK(s, cudaGetLastError());
    if (s->dual) {      /* classes of the coming tick from the headers: written through the *_next pointers */
        PveState t = s->st;
        t.klass_next = s->klass_buf[s->phase]; t.big_list_next = s->big_list_buf[s->phase]; t.big_cnt_next = s->big_cnt3;
        RT_CHECK(s, cudaMemsetAsync(s->big_cnt3, 0, 3 * sizeof(int32_t), stream));
        pve_classify_kernel<<<(s->cfg.n_envs + 127) / 128, 128, 0, stream>>>(t, s->cfg.n_envs);
        RT_CHECK(s, cudaGetLastError());
    }
#else
    (void)stream;
    emul_gsum(s->st.n_ctrl, s->gsum, s->gsum + G, s->gsum + 2 * (size_t)G, s->cfg.n_envs, G);
#endif
    return PVE_OK;
}

/* capacity classes (compile-time shared-memory layouts): veh_cap / agent_cap are rounded up to one */
#define PVE_CLASSES(X) X(96, 48) X(96, 64) X(128, 80) X(128, 96) X(192, 128) X(384, 320) X(576, 416)

static bool pick_class(int veh_cap, int agent_cap, int *VC, int *AC, size_t *smem) {
#define X(vc, ac) if (veh_cap <= vc && agent_cap <= ac) { *VC = vc; *AC = ac; *smem = PveLayout<vc, ac>::BYTES; return true; }
    PVE_CLASSES(X)
#undef X
    return false;
}

/* the arrivals argument of the step kernels: the spawn table, or the Poisson generator */
template <bool POI>
static typename PveArrivalsT<POI>::type arrivals_arg(const pve_scene *s) {
    if constexpr (POI) return s->poi;
    else return s->spawn_tick;
}

#ifndef PVE_HOST_EMULATION
template <int NT, int VC, int AC, bool SRC, bool POI>
static cudaError_t launch_variant(pve_scene *s, const float *actions, const pve_outputs &O, pve_stream_t stream) {
    static bool attr_set[16] = {false};
    int dev = s->device & 15;
    if (!attr_set[dev]) {
        cudaError_t e = cudaFuncSetAttribute(pve_step_kernel<NT, VC, AC, SRC, POI>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)(PveLayout<VC, AC>::BYTES + s->smem_pad));
        if (e != cudaSuccess) return e;
        attr_set[dev] = true;
    }
    pve_step_kernel<NT, VC, AC, SRC, POI><<<s->cfg.n_envs, NT, PveLayout<VC, AC>::BYTES + s->smem_pad, stream>>>(
        s->prm, s->st, O, arrivals_arg<POI>(s), actions, s->phase);
    return cudaGetLastError();
}
/* dual mode: the small kernel (96 threads, class PVE_SMALL_VC / PVE_SMALL_AC: more intersections resident per SM) on
 * the caller's stream and, concurrently on the side stream, the big kernel for the intersections that do not fit */
#ifndef PVE_SMALL_VC
#define PVE_SMALL_VC 96
#define PVE_SMALL_AC 64
#endif
#ifndef PVE_SMALL_NT
#define PVE_SMALL_NT 96
#endif
template <int VC, int AC, bool SRC, bool POI>
static cudaError_t launch_dual(pve_scene *s, const float *actions, const pve_outputs &O, pve_stream_t stream) {
    static bool attr_set[16] = {false};
    int dev = s->device & 15;
    const size_t smem_small = PveLayout<PVE_SMALL_VC, PVE_SMALL_AC>::BYTES, smem_big = PveLayout<VC, AC>::BYTES;
    cudaError_t e;
    if (!attr_set[dev]) {
        e = cudaFuncSetAttribute(pve_step_kernel<PVE_SMALL_NT, PVE_SMALL_VC, PVE_SMALL_AC, SRC, POI>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(smem_small + s->smem_pad));
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(pve_step_big_kernel<128, VC, AC, SRC, POI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_big);
        if (e != cudaSuccess) return e;
        attr_set[dev] = true;
    }
    const int big_grid = s->cfg.n_envs < 148 ? s->cfg.n_envs : 148;
    if (s->dual_pdl) {
        /* Experiment (env PVE_DUAL_PDL=1), measured slower than the fork / join over the side stream (0.0816 vs 0.0774 ms
         * per tick): one stream, no events: the big kernel first, the small kernel as its programmatic dependent -- it
         * starts when every CTA of the big kernel has executed griddepcontrol.launch_dependents and waits for the big
         * kernel's completion only at its own end (griddepcontrol.wait), so the stream's next kernel is ordered after
         * both. */
        pve_step_big_kernel<128, VC, AC, SRC, POI><<<big_grid, 128, smem_big, stream>>>(s->prm, s->st, O, arrivals_arg<POI>(s), actions, s->phase);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof cfg);
        cfg.gridDim = dim3((unsigned)s->cfg.n_envs); cfg.blockDim = dim3(PVE_SMALL_NT);
        cfg.dynamicSmemBytes = smem_small + s->smem_pad; cfg.stream = stream;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        const typename PveArrivalsT<POI>::type sp_arg = arrivals_arg<POI>(s);
        return cudaLaunchKernelEx(&cfg, pve_step_kernel<PVE_SMALL_NT, PVE_SMALL_VC, PVE_SMALL_AC, SRC, POI>, s->prm, s->st, O, sp_arg, actions, (int)s->phase);
    }
    if ((e = cudaEventRecord(s->ev_fork, stream)) != cudaSuccess) return e;
    if ((e = cudaStreamWaitEvent(s->side, s->ev_fork, 0)) != cudaSuccess) return e;
    pve_step_big_kernel<128, VC, AC, SRC, POI><<<big_grid, 128, smem_big, s->side>>>(s->prm, s->st, O, arrivals_arg<POI>(s), actions, s->phase);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    if ((e = cudaEventRecord(s->ev_join, s->side)) != cudaSuccess) return e;
    pve_step_kernel<PVE_SMALL_NT, PVE_SMALL_VC, PVE_SMALL_AC, SRC, POI><<<s->cfg.n_envs, PVE_SMALL_NT, smem_small + s->smem_pad, stream>>>(
        s->prm, s->st, O, arrivals_arg<POI>(s), actions, s->phase);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    return cudaStreamWaitEvent(stream, s->ev_join, 0);
}

/* the instantiation that also writes pve_outputs.nbr_src and the factored observation only when the caller asks for
 * one of them; the Poisson instantiation only in Poisson mode */
static bool wants_src(const pve_outputs &O) { return O.nbr_src != nullptr || O.obs_src != nullptr; }
template <int NT, int VC, int AC>
static cudaError_t launch_one(pve_scene *s, const float *actions, const pve_outputs &O, pve_stream_t stream) {
    if (s->poisson)
        return wants_src(O) ? launch_variant<NT, VC, AC, true, true>(s, actions, O, stream)
                            : launch_variant<NT, VC, AC, false, true>(s, actions, O, stream);
    return wants_src(O) ? launch_variant<NT, VC, AC, true, false>(s, actions, O, stream)
                     : launch_variant<NT, VC, AC, false, false>(s, actions, O, stream);
}
template <int VC, int AC>
static cudaError_t launch_dual_any(pve_scene *s, const float *actions, const pve_outputs &O, pve_stream_t stream) {
    if (s->poisson)
        return wants_src(O) ? launch_dual<VC, AC, true, true>(s, actions, O, stream) : launch_dual<VC, AC, false, true>(s, actions, O, stream);
    return wants_src(O) ? launch_dual<VC, AC, true, false>(s, actions, O, stream) : launch_dual<VC, AC, false, false>(s, actions, O, stream);
}
#endif

#ifndef PVE_HOST_EMULATION
/* lane_num = 4 / 8: the step kernel of one arrival source; SRC: the instantiation that writes pve_outputs.nbr_src.
 * S holds the stored rows of the tick's start in row0[0] (see pve4_step_block). */
template <bool POI, bool SRC>
static cudaError_t launch_kernel4(pve_scene *s, const PveState &S, const float *actions, const pve_outputs &O, pve_stream_t stream) {
    static bool attr_set[16] = {false};
    /* capacity class 64 (lists and vehicle slots of <= 64 entries): half the shared memory, twice the resident warps */
    const bool small = s->prm.VC <= 64;
    const size_t smem = (small ? sizeof(Pve4SmemT<64>) : sizeof(Pve4SmemT<128>)) * PVE4_WARPS;
    cudaError_t e;
    if (!attr_set[s->device & 15]) {
        if ((e = cudaFuncSetAttribute(pve4_step_kernel<4, 128, POI, SRC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(Pve4SmemT<128>) * PVE4_WARPS))) != cudaSuccess) return e;
        if ((e = cudaFuncSetAttribute(pve4_step_kernel<8, 128, POI, SRC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(Pve4SmemT<128>) * PVE4_WARPS))) != cudaSuccess) return e;
        if ((e = cudaFuncSetAttribute(pve4_step_kernel<4, 64, POI, SRC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(Pve4SmemT<64>) * PVE4_WARPS))) != cudaSuccess) return e;
        if ((e = cudaFuncSetAttribute(pve4_step_kernel<8, 64, POI, SRC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(Pve4SmemT<64>) * PVE4_WARPS))) != cudaSuccess) return e;
        attr_set[s->device & 15] = true;
    }
    const int grid = (s->cfg.n_envs + PVE4_WARPS - 1) / PVE4_WARPS;
    const typename PveArrivalsT<POI>::type arr = arrivals_arg<POI>(s);
    if (s->lane_num == 4 && small)
        pve4_step_kernel<4, 64, POI, SRC><<<grid, 32 * PVE4_WARPS, smem, stream>>>(s->prm4, S, O, arr, nullptr, actions, s->off4);
    else if (s->lane_num == 4)
        pve4_step_kernel<4, 128, POI, SRC><<<grid, 32 * PVE4_WARPS, smem, stream>>>(s->prm4, S, O, arr, nullptr, actions, s->off4);
    else if (small)
        pve4_step_kernel<8, 64, POI, SRC><<<grid, 32 * PVE4_WARPS, smem, stream>>>(s->prm4, S, O, arr, s->draws, actions, s->off4);
    else
        pve4_step_kernel<8, 128, POI, SRC><<<grid, 32 * PVE4_WARPS, smem, stream>>>(s->prm4, S, O, arr, s->draws, actions, s->off4);
    return cudaGetLastError();
}
#endif

/* lane_num = 4 / 8: offsets, the step, and the group sums that pve_next_agent_total reads.  The stored rows are
 * row0[phase].  A step that writes nbr_src leaves them untouched, writes the next tick's rows into row0[phase ^ 1] and
 * flips the phase, so that row0[phase ^ 1] holds the rows it read until the next step (as on 12 lanes); a step without
 * nbr_src rewrites row0[phase] in place.  n_ctrl is rewritten in place too: it does not follow the phase here. */
static int32_t launch_step4(pve_scene *s, const float *actions, const pve_outputs &O, pve_stream_t stream) {
    const int B = s->cfg.n_envs;
    const bool src = O.nbr_src != nullptr;      /* check_factored refuses the other SRC outputs on 4 / 8 lanes */
    PveState S = s->st;
    S.row0[0] = s->st.row0[s->phase]; S.row0[1] = s->st.row0[s->phase ^ 1];
#ifndef PVE_HOST_EMULATION
    if (s->profiling) RT_CHECK(s, cudaEventRecord(s->ev[0], stream));
    pve4_offsets_kernel<<<1, 1024, 0, stream>>>(s->st.n_ctrl, s->off4, B);
    RT_CHECK(s, cudaGetLastError());
    if (s->poisson) RT_CHECK(s, (src ? launch_kernel4<true, true>(s, S, actions, O, stream) : launch_kernel4<true, false>(s, S, actions, O, stream)));
    else RT_CHECK(s, (src ? launch_kernel4<false, true>(s, S, actions, O, stream) : launch_kernel4<false, false>(s, S, actions, O, stream)));
    if (s->profiling) RT_CHECK(s, cudaEventRecord(s->ev[1], stream));
    const int G = s->n_groups;
    pve_gsum_kernel<<<(G + 127) / 128, 128, 0, stream>>>(s->st.n_ctrl, s->gsum, s->gsum + G, s->gsum + 2 * (size_t)G, B, G);
    RT_CHECK(s, cudaGetLastError());
#else
    (void)stream;
    int64_t run = 0;
    for (int b = 0; b < B; ++b) { s->off4[b] = run; run += s->st.n_ctrl[b]; }
    s->off4[B] = run;
    Pve4Smem *M = new (std::nothrow) Pve4Smem;
    if (!M) return PVE_ENOMEM;
#define STEP4(NLN, POI, ARR, DRAWS)                                                                              \
    (src ? pve4_step_block<NLN, POI, true>(s->prm4, S, O, ARR, DRAWS, actions, b, *M, s->off4[b])               \
         : pve4_step_block<NLN, POI, false>(s->prm4, S, O, ARR, DRAWS, actions, b, *M, s->off4[b]))
    for (int b = 0; b < B; ++b) {
        memset(M, 0xA5, sizeof *M);           /* poison: catches reads of unwritten shared memory */
        if (s->poisson && s->lane_num == 4) STEP4(4, true, s->poi, nullptr);
        else if (s->poisson) STEP4(8, true, s->poi, nullptr);
        else if (s->lane_num == 4) STEP4(4, false, s->spawn_tick, nullptr);
        else STEP4(8, false, s->spawn_tick, s->draws);
    }
#undef STEP4
    delete M;
    emul_gsum(s->st.n_ctrl, s->gsum, s->gsum + s->n_groups, s->gsum + 2 * (size_t)s->n_groups, B, s->n_groups);
#endif
    if (src) s->phase ^= 1;
    return PVE_OK;
}

/* the factored observation (pve_outputs.row0_out / prev_row0 / obs_src): all three fields or none, 12-lane only */
static int32_t check_factored(pve_scene *s, const pve_outputs &O) {
    const int n = (O.row0_out != nullptr) + (O.prev_row0 != nullptr) + (O.obs_src != nullptr);
    if (n != 0 && n != 3) {
        snprintf(s->err, sizeof s->err, "the factored observation needs all of row0_out, prev_row0 and obs_src (%d of 3 set)", n);
        return PVE_EINVAL;
    }
    if (n != 0 && s->lane_num != 12) {
        snprintf(s->err, sizeof s->err, "lane_num = %d: the factored observation (row0_out / prev_row0 / obs_src) exists for "
                                        "the 12-lane intersection only", s->lane_num);
        return PVE_EINVAL;
    }
    return PVE_OK;
}

static int32_t launch_step(pve_scene *s, const float *actions, const pve_outputs &O_in, pve_stream_t stream) {
    const int VCc = s->prm.VC, ACc = s->prm.AC;
    pve_outputs O = O_in;
    const int32_t rc = check_factored(s, O);
    if (rc != PVE_OK) return rc;
    if (s->lane_num != 12) return launch_step4(s, actions, O, stream);
    if (s->exp_no_obs) O.obs = nullptr;          /* experiment knob (env PVE_EXPERIMENT_NO_OBS): what the observation traffic costs */
#ifndef PVE_HOST_EMULATION
    if (s->cfg.n_envs >= 1024) {                 /* small batches fit in one wave: order is irrelevant */
        if (s->order_age < 0 || s->order_age >= 32) {
            pve_order_kernel<<<1, 1024, 0, stream>>>(s->st.n_ctrl, s->order, s->cfg.n_envs);
            RT_CHECK(s, cudaGetLastError());
            s->order_age = 0;
        }
        s->order_age += 1;
        s->st.order = s->order;
    } else {
        s->st.order = nullptr;
    }
    if (s->profiling) RT_CHECK(s, cudaEventRecord(s->ev[0], stream));
    bool done = false;
    if (s->dual) {
        done = true;
        if (VCc == 192) RT_CHECK(s, (launch_dual_any<192, 128>(s, actions, O, stream)));
        else if (ACc == 96) RT_CHECK(s, (launch_dual_any<128, 96>(s, actions, O, stream)));
        else RT_CHECK(s, (launch_dual_any<128, 80>(s, actions, O, stream)));
    }
#define X(vc, ac)                                                                              \
    if (!done && VCc == vc && ACc == ac) {                                                     \
        done = true;                                                                           \
        if (s->threads == 64) RT_CHECK(s, (launch_one<64, vc, ac>(s, actions, O, stream)));    \
        else if (s->threads == 96) RT_CHECK(s, (launch_one<96, vc, ac>(s, actions, O, stream))); \
        else if (s->threads == 256) RT_CHECK(s, (launch_one<256, vc, ac>(s, actions, O, stream))); \
        else if (s->threads == 512) RT_CHECK(s, (launch_one<512, vc, ac>(s, actions, O, stream))); \
        else RT_CHECK(s, (launch_one<128, vc, ac>(s, actions, O, stream)));                    \
    }
    PVE_CLASSES(X)
#undef X
    if (!done) { snprintf(s->err, sizeof s->err, "internal: no kernel for class %d/%d", VCc, ACc); return PVE_EINVAL; }
    if (s->profiling) RT_CHECK(s, cudaEventRecord(s->ev[1], stream));
#else
    (void)stream;
    const int B = s->cfg.n_envs;
    unsigned char *smem = (unsigned char *)aligned_alloc(64, (s->smem_bytes + 63) / 64 * 64);
    if (!smem) return PVE_ENOMEM;
    bool done = false;
#define X(vc, ac)                                                                              \
    if (!done && VCc == vc && ACc == ac) {                                                     \
        done = true;                                                                           \
        for (int b = 0; b < B; ++b) {                                                          \
            memset(smem, 0xA5, s->smem_bytes); /* poison: catches reads of unwritten shared memory */ \
            if (s->poisson) pve_step_block<64, vc, ac, true, true>(s->prm, s->st, O, s->poi, actions, s->phase, b, smem, nullptr); \
            else pve_step_block<64, vc, ac, true, false>(s->prm, s->st, O, s->spawn_tick, actions, s->phase, b, smem, nullptr); \
        }                                                                                      \
    }
    PVE_CLASSES(X)
#undef X
    free(smem);
    if (!done) return PVE_EINVAL;
#endif
    s->phase ^= 1;
    s->rot = (s->rot + 1) % 3;
    set_rotation(s);
    return PVE_OK;
}

static pve_outputs null_outputs() {
    pve_outputs o;
    memset(&o, 0, sizeof o);
    return o;
}

/* =============================================================================================
 * C ABI
 * =========================================================================================== */
extern "C" {

const char *pve_backend(void) { return PVE_BACKEND; }

int32_t pve_config_bytes(void) { return (int32_t)sizeof(pve_config); }

int32_t pve_default_config(pve_config *c, int32_t n_envs, double vm) {
    if (!c) return PVE_EINVAL;
    memset(c, 0, sizeof *c);
    const double dis_ctl = 150, cw = 2.5;
    c->n_envs = n_envs; c->veh_cap = 160; c->agent_cap = 96; c->threads = 0;
    c->out_cap = (int64_t)n_envs * 96;
    c->dt = 0.1; c->dt2 = pow(0.1, 2);
    c->vm = vm; c->vM = 13; c->am = -3; c->aM = 3; c->v0 = 10; c->collision_thr = 2;
    c->lane_cw = cw;
    c->lane_in = dis_ctl - 6 * cw;
    c->lane_len[0] = 3.1415 / 2 * 7 * cw; c->lane_len[1] = 12 * cw; c->lane_len[2] = 3.1415 / 2 * cw;
    c->remove_p = -dis_ctl + (int)((12 + 1) / 2) * cw;
    const double cita = (2 * sqrt(10.0) - 6) * cw;
    const double alpha = atan((6 * cw + cita) / (3 * cw));
    const double beta = M_PI / 2 - alpha;
    const double gama = atan((sqrt(13.0) * cw) / (6 * cw));
    const double gama2 = M_PI / 2 - gama;
    /* straight ego (TIS:733-766) */
    c->vd_a1[1][0] = 3 * cw;         c->vd_a2[1][0] = 0;     c->vd_b[1][0] = 9 * cw;
    c->vd_a1[1][1] = beta * 7 * cw;  c->vd_a2[1][1] = 0;     c->vd_b[1][1] = 6 * cw + cita;
    c->vd_a1[1][2] = alpha * 7 * cw; c->vd_a2[1][2] = 0;     c->vd_b[1][2] = 6 * cw - cita;
    c->vd_a1[1][3] = 9 * cw;         c->vd_a2[1][3] = 0;     c->vd_b[1][3] = 3 * cw;
    /* left-turn ego (TIS:771-799) */
    c->vd_a1[0][0] = 6 * cw;         c->vd_a2[0][0] = cita;  c->vd_b[0][0] = alpha * 7 * cw;
    c->vd_a1[0][1] = gama * 7 * cw;  c->vd_a2[0][1] = 0;     c->vd_b[0][1] = gama2 * 7 * cw;
    c->vd_a1[0][2] = gama2 * 7 * cw; c->vd_a2[0][2] = 0;     c->vd_b[0][2] = gama * 7 * cw;
    c->vd_a1[0][3] = 6 * cw;         c->vd_a2[0][3] = -cita; c->vd_b[0][3] = beta * 7 * cw;
    for (int k = 0; k < 4; ++k) {
        const double rot = 3.141593 / 2 * k;
        c->rot_cos[k] = cos(rot); c->rot_sin[k] = sin(rot);
    }
    return PVE_OK;
}

const char *pve_last_error(const pve_scene *s) { return s ? s->err : "null handle"; }

void pve_destroy(pve_scene *s) {
    if (!s) return;
    rt_free(s->st.hdr); rt_free(s->st.p); rt_free(s->st.v); rt_free(s->st.a); rt_free(s->st.js);
    rt_free(s->st.meta); rt_free(s->st.row0[0]); rt_free(s->st.row0[1]);
    rt_free(s->n_ctrl_buf[0]); rt_free(s->n_ctrl_buf[1]); rt_free(s->st.n_veh); rt_free(s->st.stats); rt_free(s->gsum); rt_free(s->order);
    rt_free(s->actions_dev); rt_free(s->counters_dev); rt_free(s->off4);
    rt_host_free(s->pinned_i32); rt_host_free(s->pinned_gs);
    rt_free(s->klass_buf[0]); rt_free(s->klass_buf[1]); rt_free(s->big_list_buf[0]); rt_free(s->big_list_buf[1]);
    rt_free(s->big_cnt3);
    rt_free(s->clock_dev); rt_free(s->pend_dev);
#ifndef PVE_HOST_EMULATION
    for (int i = 0; i < 3; ++i) if (s->ev[i]) cudaEventDestroy(s->ev[i]);
    if (s->side) cudaStreamDestroy(s->side);
    if (s->a_ready) {
        cudaStreamDestroy(s->s_in); cudaStreamDestroy(s->s_out); cudaStreamDestroy(s->s_cnt); cudaFreeHost(s->a_total);
        for (int i = 0; i < PVE_ASYNC_SLOTS; ++i) {
            cudaEventDestroy(s->a_in[i]); cudaEventDestroy(s->a_k[i]); cudaEventDestroy(s->a_cnt[i]); cudaEventDestroy(s->a_done[i]);
            cudaFree(s->a_act[i]);
        }
    }
    if (s->ev_fork) cudaEventDestroy(s->ev_fork);
    if (s->ev_join) cudaEventDestroy(s->ev_join);
#endif
    delete s;
}

int32_t pve_create(const pve_config *cfg, int32_t device, pve_scene **out) {
    if (!cfg || !out) return PVE_EINVAL;
    *out = nullptr;
    pve_scene *s = new (std::nothrow) pve_scene();
    if (!s) return PVE_ENOMEM;
    memset(s, 0, sizeof *s);
    *out = s;                       /* returned even on failure so that pve_last_error works */
    s->cfg = *cfg;
    s->device = device;
    s->next_total = -1;
    const int B = cfg->n_envs;
    int VC = 0, AC = 0;
    if (B <= 0 || cfg->veh_cap <= 0 || cfg->agent_cap <= 0 || cfg->agent_cap > cfg->veh_cap || cfg->out_cap < 0 ||
        !pick_class(cfg->veh_cap, cfg->agent_cap, &VC, &AC, &s->smem_bytes)) {
        snprintf(s->err, sizeof s->err, "invalid config: n_envs=%d veh_cap=%d agent_cap=%d (largest class is 576/416)",
                 B, cfg->veh_cap, cfg->agent_cap);
        return PVE_EINVAL;
    }
    s->lane_num = (cfg->lane_num == 4 || cfg->lane_num == 8) ? cfg->lane_num : 12;
    if (cfg->lane_num != 0 && cfg->lane_num != 12 && cfg->lane_num != 4 && cfg->lane_num != 8) {
        snprintf(s->err, sizeof s->err, "lane_num must be 12, 8 or 4 (got %d)", cfg->lane_num);
        return PVE_EINVAL;
    }
    if (s->lane_num != 12) {
        if (VC > PVE4_LC) {
            snprintf(s->err, sizeof s->err, "lane_num = %d holds at most %d vehicles per intersection", s->lane_num, PVE4_LC);
            return PVE_EINVAL;
        }
        /* two capacity classes on this path: 64/64 and 128/>=96 */
        if (cfg->veh_cap <= 64) { VC = 64; AC = 64; s->smem_bytes = sizeof(Pve4SmemT<64>); }
        else { VC = 128; AC = AC < 96 ? 96 : AC; s->smem_bytes = sizeof(Pve4Smem); }
    }
    s->cfg.veh_cap = VC;          /* rounded up to the capacity class; see pve_veh_cap() */
    s->cfg.agent_cap = AC;
    /* default CTA size: 128 threads for the small classes (V ~ 76 vehicles per intersection), 512 for the large ones
     * (stress: V ~ 345, 1 600 virtual-lane entries; two CTAs per SM at 64 registers = 32 warps per SM.  Measured per
     * tick of 4 096 stress intersections: 128 threads 0.766 ms, 256: 0.586, 512: 0.487) */
    s->threads = cfg->threads == 0 ? (VC >= 384 ? 512 : 128) : cfg->threads;
#ifndef PVE_HOST_EMULATION
    /* dual mode for the classes 128/80, 128/96 and 192/128 with the default CTA size (env PVE_DUAL=0 turns it off) */
    s->dual = (cfg->threads == 0 && (VC == 128 || VC == 192) && s->lane_num == 12) ? 1 : 0;
    if (const char *d = getenv("PVE_DUAL")) s->dual = s->dual && atoi(d) != 0;
    s->dual_pdl = 0;      /* experiment knob: 1 = one stream, the small kernel as the big kernel's programmatic dependent */
    if (const char *d = getenv("PVE_DUAL_PDL")) s->dual_pdl = atoi(d) != 0;
#endif
    if (const char *pad = getenv("PVE_SMEM_PAD")) s->smem_pad = (size_t)atoi(pad);
    s->exp_no_obs = getenv("PVE_EXPERIMENT_NO_OBS") != nullptr;
    s->host_zerocopy = 1;
    if (const char *zc = getenv("PVE_HOST_ZEROCOPY")) s->host_zerocopy = atoi(zc);
    if (s->threads != 64 && s->threads != 96 && s->threads != 128 && s->threads != 256 && s->threads != 512) {
        snprintf(s->err, sizeof s->err, "threads must be 0, 64, 96, 128, 256 or 512");
        return PVE_EINVAL;
    }
    PveParams &P = s->prm;
    memset(&P, 0, sizeof P);
    P.dt = cfg->dt; P.dt2 = cfg->dt2; P.vm = cfg->vm; P.vM = cfg->vM; P.am = cfg->am; P.aM = cfg->aM;
    P.v0 = cfg->v0; P.thr = cfg->collision_thr; P.lane_in = cfg->lane_in; P.remove_p = cfg->remove_p;
    P.lane_cw = cfg->lane_cw; P.abs_am = fabs(cfg->am); P.two_abs_am = 2 * fabs(cfg->am);     /* TIS:1513-1514 */
    P.r_abs_am = 1.0 / P.abs_am; P.r_two_abs_am = 1.0 / P.two_abs_am;
    P.aspan = (double)(cfg->aM - cfg->am);                                                     /* TIS:319 */
    for (int m = 0; m < 3; ++m) { P.lane_len[m] = cfg->lane_len[m]; P.spawn_p[m] = cfg->lane_in + cfg->lane_len[m]; }  /* TIS:395 */
    memcpy(P.vd_a1, cfg->vd_a1, sizeof P.vd_a1); memcpy(P.vd_a2, cfg->vd_a2, sizeof P.vd_a2);
    memcpy(P.vd_b, cfg->vd_b, sizeof P.vd_b);
    memcpy(P.rot_cos, cfg->rot_cos, sizeof P.rot_cos); memcpy(P.rot_sin, cfg->rot_sin, sizeof P.rot_sin);
    P.f_cw = (float)P.lane_cw; P.f_thr = (float)P.thr;
    for (int m = 0; m < 3; ++m) { P.f_len[m] = (float)P.lane_len[m]; P.f_rq[m] = (float)(3.141593 / 2 / P.lane_len[m]); }   /* TIS:1259 */
    for (int k = 0; k < 4; ++k) { P.f_rc[k] = (float)P.rot_cos[k]; P.f_rs[k] = (float)P.rot_sin[k]; }
    memcpy(P.l2l, kLane2Lane, sizeof P.l2l);
    memset(P.rev_dir, -1, sizeof P.rev_dir);
    for (int L = 0; L < PVE_NLANE; ++L) {
        int n = 0;
        for (int d = 0; d < PVE_NLANE; ++d)
            for (int k = 0; k < 4; ++k)
                if (kLane2Lane[d][k] == L && n < 4) { P.rev_dir[L][n] = (int8_t)d; P.rev_k[L][n] = (int8_t)k; ++n; }
        if ((L % 3 != 2 && n != 4) || (L % 3 == 2 && n != 0)) {
            snprintf(s->err, sizeof s->err, "internal: conflict table is not 4-regular");
            return PVE_EINVAL;
        }
    }
    if (s->lane_num != 12) {
        static const int8_t kDir4[PVE4_NL][3] = {{6, 7, 8}, {0, 1, 2}, {9, 10, 11}, {3, 4, 5}};                  /* TIS:73-78 */
        static const int8_t kL2L4[PVE4_ND][7] = {                                                                /* TIS:58-71 */
            {10, 6, 9, 3, 7, 4, 8}, {10, 6, 3, 4, 9, 5, -1}, {6, 10, -1, -1, -1, -1, -1},
            {1, 9, 0, 6, 10, 7, 11}, {1, 9, 6, 7, 0, 8, -1}, {9, 1, -1, -1, -1, -1, -1},
            {4, 0, 3, 9, 1, 10, 2}, {4, 0, 9, 10, 3, 11, -1}, {0, 4, -1, -1, -1, -1, -1},
            {7, 3, 6, 0, 4, 1, 5}, {7, 3, 0, 1, 6, 2, -1}, {3, 7, -1, -1, -1, -1, -1}};
        static const int8_t kDir8[PVE4_MAXNL][3] = {{0, 1, -1}, {-1, 2, 3}, {4, 5, -1}, {-1, 6, 7},             /* TIS:136-145 */
                                                    {8, 9, -1}, {-1, 10, 11}, {12, 13, -1}, {-1, 14, 15}};
        static const int8_t kL2L8[PVE4_MAXND][7] = {                                                             /* TIS:107-123 */
            {14, 4, 13, 12, 9, 10, 5}, {14, 13, 8, 4, 5, 6, 12}, {14, 13, 8, 4, 5, 6, 7}, {14, -1, -1, -1, -1, -1, -1},
            {2, 8, 1, 0, 13, 14, 9}, {2, 1, 12, 8, 9, 10, 0}, {2, 1, 12, 8, 9, 10, 11}, {2, -1, -1, -1, -1, -1, -1},
            {6, 12, 5, 4, 1, 2, 13}, {6, 5, 0, 12, 13, 14, 4}, {6, 5, 0, 12, 13, 14, 15}, {6, -1, -1, -1, -1, -1, -1},
            {10, 0, 9, 8, 5, 6, 1}, {10, 9, 4, 0, 1, 2, 8}, {10, 9, 4, 0, 1, 2, 3}, {10, -1, -1, -1, -1, -1, -1}};
        const bool four = s->lane_num == 4;
        const int nl = four ? PVE4_NL : PVE4_MAXNL, nd = four ? PVE4_ND : PVE4_MAXND;
        Pve4Params &Q = s->prm4;
        memset(&Q, 0, sizeof Q);
        Q.dt = cfg->dt; Q.dt2 = cfg->dt2; Q.vm = cfg->vm; Q.vM = cfg->vM; Q.am = cfg->am; Q.aM = cfg->aM; Q.v0 = cfg->v0;
        Q.thr = cfg->collision_thr; Q.lane_in = cfg->lane_in; Q.remove_p = cfg->remove_p; Q.cw = cfg->lane_cw;
        Q.abs_am = fabs(cfg->am); Q.two_abs_am = 2 * fabs(cfg->am); Q.aspan = (double)(cfg->aM - cfg->am);
        for (int m = 0; m < 3; ++m) Q.L[m] = cfg->lane_len[m];
        memcpy(Q.T, cfg->n4_T, sizeof Q.T); memcpy(Q.C, cfg->n4_C, sizeof Q.C); memcpy(Q.C2, cfg->n4_C2, sizeof Q.C2);
        Q.rw_k = cfg->n4_rw[0]; Q.rw_a = cfg->n4_rw[1]; Q.rw_b = cfg->n4_rw[2];
        memset(Q.dir, -1, sizeof Q.dir);
        for (int i = 0; i < nl; ++i) for (int m = 0; m < 3; ++m) Q.dir[i][m] = four ? kDir4[i][m] : kDir8[i][m];
        memset(Q.l2l_pos, -1, sizeof Q.l2l_pos);
        for (int d = 0; d < nd; ++d) {
            for (int k = 0; k < 7; ++k) {
                const int r = four ? kL2L4[d][k] : kL2L8[d][k];
                if (r >= 0) Q.l2l_pos[d][r] = (int8_t)k;
            }
            Q.l2l_1[d] = four ? kL2L4[d][1] : kL2L8[d][1];
        }
        for (int i = 0; i < PVE4_MAXNL; ++i) { Q.int8[i][0] = (int8_t)((i & 1) ? 1 : 0); Q.int8[i][1] = (int8_t)((i & 1) ? 2 : 1); }   /* TIS:125-134 */
        Q.ntype = four ? 3 : 4;
        for (int i = 0; i < nl; ++i) if (i == 2 || i == 5 || i == 8 || i == 11) Q.am_mask |= 1 << i;             /* TIS:1519 */
        Q.B = B; Q.VC = VC; Q.K = 0; Q.zero_unctl = cfg->zero_uncontrolled ? 1 : 0; Q.out_cap = cfg->out_cap;
    }
    P.B = B; P.VC = VC; P.AC = AC; P.K = 0; P.out_cap = cfg->out_cap;
    s->st.small_vc = 0; s->st.small_ac = 0;
    P.zero_unctl = cfg->zero_uncontrolled ? 1 : 0;
#ifndef PVE_HOST_EMULATION
    RT_CHECK(s, cudaSetDevice(device));
#endif
    const size_t nv = (size_t)B * VC;
    RT_CHECK(s, rt_alloc((void **)&s->st.hdr, sizeof(pve_env_header) * (size_t)B));
    RT_CHECK(s, rt_alloc((void **)&s->st.p, sizeof(double) * nv));
    RT_CHECK(s, rt_alloc((void **)&s->st.v, sizeof(double) * nv));
    RT_CHECK(s, rt_alloc((void **)&s->st.a, sizeof(double) * nv));
    RT_CHECK(s, rt_alloc((void **)&s->st.js, sizeof(double) * nv));
    RT_CHECK(s, rt_alloc((void **)&s->st.meta, sizeof(pve_veh_meta) * nv));
    RT_CHECK(s, rt_alloc((void **)&s->st.row0[0], sizeof(float) * nv * PVE_OBS_W));
    RT_CHECK(s, rt_alloc((void **)&s->st.row0[1], sizeof(float) * nv * PVE_OBS_W));
    RT_CHECK(s, rt_alloc((void **)&s->n_ctrl_buf[0], sizeof(int32_t) * (size_t)B));
    RT_CHECK(s, rt_alloc((void **)&s->n_ctrl_buf[1], sizeof(int32_t) * (size_t)B));
    s->st.n_ctrl = s->n_ctrl_buf[0]; s->st.n_ctrl_next = s->n_ctrl_buf[1];
    RT_CHECK(s, rt_alloc((void **)&s->st.n_veh, sizeof(int32_t) * (size_t)B));
    RT_CHECK(s, rt_alloc((void **)&s->st.stats, sizeof(double) * (size_t)B * PVE_NSTAT));
    RT_CHECK(s, rt_alloc((void **)&s->order, sizeof(int32_t) * (size_t)B));
    if (s->lane_num != 12) RT_CHECK(s, rt_alloc((void **)&s->off4, sizeof(int64_t) * ((size_t)B + 1)));
    s->order_age = -1;
#ifndef PVE_HOST_EMULATION
    if (s->dual) {
        s->st.small_vc = PVE_SMALL_VC; s->st.small_ac = PVE_SMALL_AC;
        for (int i = 0; i < 2; ++i) {
            RT_CHECK(s, rt_alloc((void **)&s->klass_buf[i], (size_t)B));
            RT_CHECK(s, rt_alloc((void **)&s->big_list_buf[i], sizeof(int32_t) * (size_t)B));
        }
        RT_CHECK(s, rt_alloc((void **)&s->big_cnt3, sizeof(int32_t) * 3));
        int prio_lo = 0, prio_hi = 0;        /* the few big CTAs take free SM slots before the queue of small ones */
        RT_CHECK(s, cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        RT_CHECK(s, cudaStreamCreateWithPriority(&s->side, cudaStreamNonBlocking, prio_hi));
        RT_CHECK(s, cudaEventCreateWithFlags(&s->ev_fork, cudaEventDisableTiming));
        RT_CHECK(s, cudaEventCreateWithFlags(&s->ev_join, cudaEventDisableTiming));
    }
#endif
    s->n_groups = (B + (1 << PVE_GROUP_SHIFT) - 1) >> PVE_GROUP_SHIFT;
    RT_CHECK(s, rt_alloc((void **)&s->gsum, sizeof(int32_t) * 3 * (size_t)s->n_groups));
    RT_CHECK(s, rt_host_alloc((void **)&s->pinned_gs, sizeof(int32_t) * (size_t)s->n_groups));
    RT_CHECK(s, rt_alloc((void **)&s->counters_dev, sizeof(double) * 16));
#ifdef PVE_PHASE_TIMING
    RT_CHECK(s, rt_alloc((void **)&s->st.dbg, sizeof(long long) * 48 * (size_t)B));
#endif
    RT_CHECK(s, rt_host_alloc((void **)&s->pinned_i32, sizeof(int32_t) * 16));
    return pve_reset(s, nullptr, 0, 0, nullptr);
}

int32_t pve_set_intention_draws(pve_scene *s, const uint8_t *draws_dev) {
    if (!s) return PVE_EINVAL;
    s->draws = draws_dev;
    return PVE_OK;
}

/* the state of a new episode from the handle's arrival source (pve_reset / pve_reset_poisson); warm_step: run the tick
 * that brings the first vehicle(s) in */
static int32_t reset_state(pve_scene *s, int32_t warmup, bool warm_step, pve_stream_t stream) {
    const int B = s->cfg.n_envs;
    const size_t nv = (size_t)B * s->cfg.veh_cap;
    s->phase = 0;
    s->rot = 0;
    s->order_age = -1;
    set_rotation(s);
    s->next_total = -1;
    RT_CHECK(s, rt_memset(s->st.p, 0, sizeof(double) * nv, stream));
    RT_CHECK(s, rt_memset(s->st.v, 0, sizeof(double) * nv, stream));
    RT_CHECK(s, rt_memset(s->st.a, 0, sizeof(double) * nv, stream));
    RT_CHECK(s, rt_memset(s->st.js, 0, sizeof(double) * nv, stream));
    RT_CHECK(s, rt_memset(s->st.meta, 0, sizeof(pve_veh_meta) * nv, stream));
    RT_CHECK(s, rt_memset(s->st.row0[0], 0, sizeof(float) * nv * PVE_OBS_W, stream));
    RT_CHECK(s, rt_memset(s->st.row0[1], 0, sizeof(float) * nv * PVE_OBS_W, stream));
#ifndef PVE_HOST_EMULATION
    if (s->poisson) pve_reset_kernel<true><<<(B + 127) / 128, 128, 0, stream>>>(s->st, s->poi, B, 0, warmup);
    else pve_reset_kernel<false><<<(B + 127) / 128, 128, 0, stream>>>(s->st, s->spawn_tick, B, s->prm.K, warmup);
    RT_CHECK(s, cudaGetLastError());
#else
    if (s->poisson) emul_reset<true>(s->st, s->poi, B, 0, warmup);
    else emul_reset<false>(s->st, s->spawn_tick, B, s->prm.K, warmup);
#endif
    int32_t rc = launch_gsum(s, stream);
    if (rc != PVE_OK) return rc;
    if (warm_step) {
        /* the tick that brings the first vehicle(s) in: nothing to step, nothing to emit */
        if (!s->actions_dev) RT_CHECK(s, rt_alloc((void **)&s->actions_dev, sizeof(float) * nv));
        rc = launch_step(s, s->actions_dev, null_outputs(), stream);
    }
    return rc;
}

int32_t pve_reset(pve_scene *s, const int32_t *spawn_tick_dev, int32_t K, int32_t warmup, void *stream_) {
    if (!s) return PVE_EINVAL;
    if (s->lane_num == 8 && spawn_tick_dev && K > 0 && !s->draws) {
        snprintf(s->err, sizeof s->err, "lane_num = 8: call pve_set_intention_draws before pve_reset (TIS:390 draws every new "
                                        "vehicle's intention at random; the draws are an input here)");
        return PVE_EINVAL;
    }
    s->poisson = 0;
    s->spawn_tick = spawn_tick_dev;
    s->prm.K = spawn_tick_dev ? K : 0;
    s->prm4.K = s->prm.K;
    return reset_state(s, warmup, warmup && spawn_tick_dev && K > 0, (pve_stream_t)stream_);
}

/* pve_reset_poisson (rates == nullptr: every lane at p->rate_veh_per_hour) and pve_reset_poisson_rates (rates: host
 * [n_envs][lane_num] veh/h); `fn` names the entry point in pve_last_error */
static int32_t reset_poisson(pve_scene *s, const pve_poisson *p, const double *rates, int32_t warmup, void *stream_,
                             const char *fn) {
    if (!s) return PVE_EINVAL;
    if (!p) { snprintf(s->err, sizeof s->err, "%s: null parameters", fn); return PVE_EINVAL; }
    const int B = s->cfg.n_envs, nl = s->lane_num;
    for (size_t q = 0; rates && q < (size_t)B * nl; ++q) {
        if (!(isfinite(rates[q]) && rates[q] > 0)) {
            snprintf(s->err, sizeof s->err, "%s: the rate of intersection %zu, lane %zu is %g; every rate must be finite "
                     "and > 0", fn, q / nl, q % nl, rates[q]);
            return PVE_EINVAL;
        }
    }
    const char *bad = nullptr;
    if (!rates && !(isfinite(p->rate_veh_per_hour) && p->rate_veh_per_hour > 0)) bad = "rate_veh_per_hour must be finite and > 0";
    else if (!(isfinite(p->min_headway) && p->min_headway > 0))
        bad = "min_headway must be finite and > 0 (an arrival at 0 s would read as table padding)";
    else if (p->first_env < 0) bad = "first_env must be >= 0";
    else if (p->first_env + (int64_t)B > ((int64_t)1 << 32)) bad = "first_env + n_envs must be <= 2^32 (the counter word of e)";
    else if (s->cfg.dt != 0.1) bad = "Poisson arrivals use the reference's 0.1 s clock (pve_config.dt must be 0.1)";
    if (bad) {
        snprintf(s->err, sizeof s->err, "%s: %s", fn, bad);
        return PVE_EINVAL;
    }
    pve_stream_t stream = (pve_stream_t)stream_;
    if (!s->clock_dev) {       /* the reference's clock, the same sequential additions as arrivals.reference_clock */
        const size_t n = (size_t)PVE_MAX_TICK + 1;
        double *clock = (double *)malloc(sizeof(double) * n);
        if (!clock) return PVE_ENOMEM;
        clock[0] = 0.0;
        for (size_t k = 1; k < n; ++k) clock[k] = clock[k - 1] + s->cfg.dt;
        s->poi.clock_last = clock[n - 1];
        int32_t rc = PVE_OK;
        if (rt_alloc((void **)&s->clock_dev, sizeof(double) * n) != 0 ||
            rt_alloc((void **)&s->pend_dev, sizeof(double) * 2 * PVE_NLANE * (size_t)B) != 0 ||
            rt_copy(s->clock_dev, clock, sizeof(double) * n, stream) != 0 || rt_sync(stream) != 0) {
            snprintf(s->err, sizeof s->err, "%s: could not set up the %zu-byte clock table", fn, sizeof(double) * n);
            rt_free(s->clock_dev); rt_free(s->pend_dev);
            s->clock_dev = nullptr; s->pend_dev = nullptr;
            rc = PVE_ECUDA;
        }
        free(clock);
        if (rc != PVE_OK) return rc;
    }
    PvePoisson &A = s->poi;
    A.clock = s->clock_dev;
    A.pend = s->pend_dev;
    A.mean = s->pend_dev + PVE_NLANE * (size_t)B;
    if (rates) {
        /* the means in float64 on the host, the same division as arrivals.poisson_arrivals; lanes past lane_num never
         * spawn and keep 0 */
        double *mean = (double *)calloc((size_t)B * PVE_NLANE, sizeof(double));
        if (!mean) return PVE_ENOMEM;
        for (size_t q = 0; q < (size_t)B * nl; ++q) mean[q / nl * PVE_NLANE + q % nl] = 3600.0 / rates[q];
        const int rc = rt_copy(A.mean, mean, sizeof(double) * PVE_NLANE * (size_t)B, stream) != 0 || rt_sync(stream) != 0;
        free(mean);
        if (rc) { snprintf(s->err, sizeof s->err, "%s: could not copy the rates to the device", fn); return PVE_ECUDA; }
        A.uniform_mean = 0.0;
    } else {
        A.uniform_mean = 3600.0 / p->rate_veh_per_hour;
    }
    A.min_headway = p->min_headway;
    A.key0 = (uint32_t)(p->seed & 0xFFFFFFFFu);
    A.key1 = (uint32_t)(p->seed >> 32);
    A.first_env = (uint32_t)p->first_env;
    A.nlane = s->lane_num;
    s->poisson = 1;
    s->spawn_tick = nullptr;
    s->prm.K = 0;
    s->prm4.K = 0;
    return reset_state(s, warmup, warmup != 0, stream);
}

int32_t pve_reset_poisson(pve_scene *s, const pve_poisson *p, int32_t warmup, void *stream) {
    return reset_poisson(s, p, nullptr, warmup, stream, "pve_reset_poisson");
}

int32_t pve_reset_poisson_rates(pve_scene *s, const pve_poisson *p, const double *rates_host, int32_t warmup, void *stream) {
    if (s && !rates_host) {
        snprintf(s->err, sizeof s->err, "pve_reset_poisson_rates: null rates_host");
        return PVE_EINVAL;
    }
    return reset_poisson(s, p, rates_host, warmup, stream, "pve_reset_poisson_rates");
}

int32_t pve_step(pve_scene *s, const float *actions_dev, const pve_outputs *out_dev, void *stream_) {
    if (!s || !actions_dev) return PVE_EINVAL;
    pve_stream_t stream = (pve_stream_t)stream_;
    const pve_outputs O = out_dev ? *out_dev : null_outputs();
    /* one launch per tick: every CTA derives its first output row from the group sums */
    int32_t rc = launch_step(s, actions_dev, O, stream);
    if (rc != PVE_OK) return rc;
    s->next_total = -1;
#ifndef PVE_HOST_EMULATION
    if (s->profiling) RT_CHECK(s, cudaEventRecord(s->ev[2], stream));
#endif
    return rc;
}

/* CUDA-event timing of the two kernels of the last pve_step (bench.py's roofline numbers).
 * pve_kernel_ms synchronises on the last event. */
int32_t pve_set_profiling(pve_scene *s, int32_t on) {
    if (!s) return PVE_EINVAL;
#ifndef PVE_HOST_EMULATION
    if (on && !s->ev[0])
        for (int i = 0; i < 3; ++i) RT_CHECK(s, cudaEventCreate(&s->ev[i]));
#endif
    s->profiling = on ? 1 : 0;
    return PVE_OK;
}

int32_t pve_kernel_ms(pve_scene *s, float *step_ms, float *scan_ms) {
    if (!s || !s->profiling) return PVE_EINVAL;
#ifndef PVE_HOST_EMULATION
    RT_CHECK(s, cudaEventSynchronize(s->ev[2]));
    if (step_ms) RT_CHECK(s, cudaEventElapsedTime(step_ms, s->ev[0], s->ev[1]));
    if (scan_ms) RT_CHECK(s, cudaEventElapsedTime(scan_ms, s->ev[1], s->ev[2]));
#else
    if (step_ms) *step_ms = 0.f;
    if (scan_ms) *scan_ms = 0.f;
#endif
    return PVE_OK;
}

int64_t pve_next_agent_total(pve_scene *s, void *stream_) {
    if (!s) return PVE_EINVAL;
    pve_stream_t stream = (pve_stream_t)stream_;
    if (s->next_total < 0) {
        RT_CHECK(s, rt_copy(s->pinned_gs, s->st.gs_read, sizeof(int32_t) * (size_t)s->n_groups, stream));
        RT_CHECK(s, rt_sync(stream));
        int64_t t = 0;
        for (int g = 0; g < s->n_groups; ++g) t += s->pinned_gs[g];
        s->next_total = t;
    }
    return s->next_total;
}

#ifndef PVE_HOST_EMULATION
/* true if the device can address `p` directly as host memory (cudaHostAlloc / cudaHostRegister: torch's
 * pin_memory()), which lets the kernel read or write it in place over PCIe */
static bool is_pinned_host(const void *p) {
    if (!p) return false;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
}
#endif

int32_t pve_step_host(pve_scene *s, const float *actions_host, const pve_outputs *out_dev,
                      const pve_outputs *out_host, int32_t copy_mask, void *stream_) {
    if (!s || !actions_host || !out_dev) return PVE_EINVAL;
    pve_stream_t stream = (pve_stream_t)stream_;
    const int B = s->cfg.n_envs;
    const size_t nv = (size_t)B * s->cfg.veh_cap;
    const int64_t A = pve_next_agent_total(s, stream_);
    if (A < 0) return (int32_t)A;
    if (A > s->cfg.out_cap) {
        snprintf(s->err, sizeof s->err, "tick emits %lld rows but out_cap is %lld", (long long)A, (long long)s->cfg.out_cap);
        return PVE_ESTATE;
    }
    const size_t a = (size_t)A;
    /* Zero-copy path (pinned host buffers, the normal case): the kernel reads the actions and writes the small
     * per-agent outputs in place over PCIe while it runs, instead of 1 + 9 staged copies around it.  In that
     * case those arrays of out_dev are NOT written this tick (the observations always are).
     * PVE_HOST_ZEROCOPY=0 turns it off. */
    const float *act_for_kernel = nullptr;
    pve_outputs O = *out_dev;
    bool mirrored = false;
#ifndef PVE_HOST_EMULATION
    if (s->host_zerocopy == 1 && is_pinned_host(actions_host)) act_for_kernel = actions_host;   /* 2: outputs only */
    if (s->host_zerocopy && out_host && (copy_mask & 1)) {
        const void *f[9] = {out_host->agent_offset, out_host->reward, out_host->ids, out_host->cpv, out_host->status,
                            out_host->jerk_sum, out_host->env_collisions, out_host->env_lock, out_host->env_removed};
        mirrored = true;
        for (int i = 0; i < 9; ++i) if (!f[i] || !is_pinned_host(f[i])) mirrored = false;
        if (mirrored) {
            O.agent_offset = out_host->agent_offset; O.reward = out_host->reward; O.ids = out_host->ids;
            O.cpv = out_host->cpv; O.status = out_host->status; O.jerk_sum = out_host->jerk_sum;
            O.env_collisions = out_host->env_collisions; O.env_lock = out_host->env_lock;
            O.env_removed = out_host->env_removed;
        }
    }
#endif
    if (!act_for_kernel) {
        if (!s->actions_dev) RT_CHECK(s, rt_alloc((void **)&s->actions_dev, sizeof(float) * nv));
        RT_CHECK(s, rt_copy(s->actions_dev, actions_host, sizeof(float) * nv, stream));
        act_for_kernel = s->actions_dev;
    }
    int32_t rc = launch_step(s, act_for_kernel, O, stream);
    if (rc != PVE_OK) return rc;
    s->next_total = -1;
    if (out_host && (copy_mask & 1) && !mirrored) {
#define D2H(field, bytes) \
        if (out_host->field && out_dev->field) RT_CHECK(s, rt_copy(out_host->field, out_dev->field, (bytes), stream))
        D2H(agent_offset, sizeof(int32_t) * ((size_t)B + 1));
        D2H(reward, sizeof(float) * a);
        D2H(ids, sizeof(int32_t) * 4 * a);
        D2H(cpv, sizeof(int32_t) * a);
        D2H(status, sizeof(uint8_t) * a);
        D2H(jerk_sum, sizeof(float) * a);
        D2H(env_collisions, sizeof(int32_t) * (size_t)B);
        D2H(env_lock, sizeof(int32_t) * (size_t)B);
        D2H(env_removed, sizeof(int32_t) * (size_t)B);
    }
    if (out_host && (copy_mask & 2)) {
        D2H(obs, sizeof(float) * PVE_OBS_H * PVE_OBS_W * a);
#undef D2H
    }
    RT_CHECK(s, rt_copy(s->pinned_gs, s->st.gs_read, sizeof(int32_t) * (size_t)s->n_groups, stream));
    RT_CHECK(s, rt_sync(stream));
    int64_t t = 0;
    for (int g = 0; g < s->n_groups; ++g) t += s->pinned_gs[g];
    s->next_total = t;
    return PVE_OK;
}

#ifndef PVE_HOST_EMULATION
static int32_t async_setup(pve_scene *s) {
    if (s->a_ready) return PVE_OK;
    const size_t nv = (size_t)s->cfg.n_envs * s->cfg.veh_cap;
    RT_CHECK(s, cudaStreamCreateWithFlags(&s->s_in, cudaStreamNonBlocking));
    RT_CHECK(s, cudaStreamCreateWithFlags(&s->s_out, cudaStreamNonBlocking));
    RT_CHECK(s, cudaStreamCreateWithFlags(&s->s_cnt, cudaStreamNonBlocking));
    RT_CHECK(s, rt_host_alloc((void **)&s->a_total, sizeof(int64_t) * PVE_ASYNC_SLOTS));
    for (int i = 0; i < PVE_ASYNC_SLOTS; ++i) {
        RT_CHECK(s, cudaEventCreateWithFlags(&s->a_in[i], cudaEventDisableTiming));
        RT_CHECK(s, cudaEventCreateWithFlags(&s->a_k[i], cudaEventDisableTiming));
        RT_CHECK(s, cudaEventCreateWithFlags(&s->a_cnt[i], cudaEventDisableTiming));
        RT_CHECK(s, cudaEventCreateWithFlags(&s->a_done[i], cudaEventDisableTiming));
        RT_CHECK(s, rt_alloc((void **)&s->a_act[i], sizeof(float) * nv));
    }
    s->a_ready = 1;
    return PVE_OK;
}
#endif

#ifndef PVE_HOST_EMULATION
/* copy-out of tick `seq` (enqueued one call late, when its row count has long arrived): DMA behind its kernel */
static int32_t async_copy_out(pve_scene *s, int64_t seq) {
    const int slot = (int)(seq % PVE_ASYNC_SLOTS);
    const int B = s->cfg.n_envs;
    int64_t A = s->a_rows[slot];
    if (A < 0) {                               /* the sums the previous tick's kernel sent home */
        const int prev = (int)((seq + PVE_ASYNC_SLOTS - 1) % PVE_ASYNC_SLOTS);
        RT_CHECK(s, cudaEventSynchronize(s->a_cnt[prev]));
        A = s->a_total[prev];
        s->a_rows[slot] = A;
    }
    if (A > s->cfg.out_cap) {
        snprintf(s->err, sizeof s->err, "tick emits %lld rows but out_cap is %lld", (long long)A, (long long)s->cfg.out_cap);
        return PVE_ESTATE;
    }
    const size_t a = (size_t)A;
    const pve_outputs *out_dev = &s->a_odev[slot], *out_host = &s->a_ohost[slot];
    RT_CHECK(s, cudaStreamWaitEvent(s->s_out, s->a_k[slot], 0));
#define D2HA(field, bytes) \
    if (out_host->field && out_dev->field) RT_CHECK(s, cudaMemcpyAsync(out_host->field, out_dev->field, (bytes), cudaMemcpyDeviceToHost, s->s_out))
    /* agent_offset[B+1] | env_collisions[B] | env_lock[B] | env_removed[B] in one allocation on both sides: one copy */
    const bool small_contig = out_dev->env_collisions == out_dev->agent_offset + B + 1 && out_dev->env_lock == out_dev->env_collisions + B &&
                              out_dev->env_removed == out_dev->env_lock + B && out_host->env_collisions == out_host->agent_offset + B + 1 &&
                              out_host->env_lock == out_host->env_collisions + B && out_host->env_removed == out_host->env_lock + B;
    if (small_contig) {
        D2HA(agent_offset, sizeof(int32_t) * (4 * (size_t)B + 1));
    } else {
        D2HA(agent_offset, sizeof(int32_t) * ((size_t)B + 1));
        D2HA(env_collisions, sizeof(int32_t) * (size_t)B);
        D2HA(env_lock, sizeof(int32_t) * (size_t)B);
        D2HA(env_removed, sizeof(int32_t) * (size_t)B);
    }
    D2HA(packed, sizeof(pve_agent_record) * a);
    if (s->a_mask[slot] & 2) D2HA(obs, sizeof(float) * PVE_OBS_H * PVE_OBS_W * a);
    if (s->a_mask[slot] & 4) {                 /* the factored observation: 240 instead of 784 bytes per agent */
        D2HA(row0_out, sizeof(float) * PVE_OBS_W * a);
        D2HA(prev_row0, sizeof(float) * PVE_OBS_W * a);
        D2HA(obs_src, sizeof(int16_t) * 8 * a);
    }
#undef D2HA
    RT_CHECK(s, cudaEventRecord(s->a_done[slot], s->s_out));
    s->a_copied = seq + 1;
    return PVE_OK;
}
#endif

int32_t pve_step_host_async(pve_scene *s, const float *actions_host, const pve_outputs *out_dev,
                            const pve_outputs *out_host, int32_t copy_mask, void *stream_) {
    if (!s || !actions_host || !out_dev || !out_host) return PVE_EINVAL;
#ifdef PVE_HOST_EMULATION
    (void)copy_mask; (void)stream_;
    return PVE_ESTATE;                       /* device only */
#else
    pve_stream_t stream = (pve_stream_t)stream_;
    if (!out_dev->packed || !out_host->packed || !out_dev->agent_offset || !out_host->agent_offset ||
        ((copy_mask & 2) && (!out_dev->obs || !out_host->obs))) {
        snprintf(s->err, sizeof s->err, "pve_step_host_async needs packed + agent_offset (and obs with bit1) in out_dev and out_host");
        return PVE_EINVAL;
    }
    if ((copy_mask & 4) && (!out_dev->obs_src || !out_host->row0_out || !out_host->prev_row0 || !out_host->obs_src)) {
        snprintf(s->err, sizeof s->err, "pve_step_host_async: copy_mask bit2 needs row0_out, prev_row0 and obs_src in out_dev "
                                        "and out_host");
        return PVE_EINVAL;
    }
    if (check_factored(s, *out_dev) != PVE_OK) return PVE_EINVAL;
    const int inflight = (int)(s->a_seq - s->a_waited);
    if (inflight >= PVE_ASYNC_SLOTS) {
        snprintf(s->err, sizeof s->err, "%d ticks are in flight: call pve_host_wait first", inflight);
        return PVE_ESTATE;
    }
    int32_t rc = async_setup(s);
    if (rc != PVE_OK) return rc;
    const size_t nv = (size_t)s->cfg.n_envs * s->cfg.veh_cap;
    const int slot = (int)(s->a_seq % PVE_ASYNC_SLOTS);
    /* rows of this tick: unknown (-1) when the previous tick came through here -- its kernel sends the sums home and
     * async_copy_out picks them up; otherwise the synchronous query */
    int64_t A = -1;
    if (inflight == 0 || s->next_total >= 0) {
        A = pve_next_agent_total(s, stream_);
        if (A < 0) return (int32_t)A;
    }
    /* actions: DMA on the copy-in stream, after the kernel that last read this buffer */
    RT_CHECK(s, cudaStreamWaitEvent(s->s_in, s->a_k[slot], 0));
    RT_CHECK(s, cudaMemcpyAsync(s->a_act[slot], actions_host, sizeof(float) * nv, cudaMemcpyHostToDevice, s->s_in));
    RT_CHECK(s, cudaEventRecord(s->a_in[slot], s->s_in));
    /* the kernel, after its actions have arrived and after the copy-out that last read these output buffers */
    RT_CHECK(s, cudaStreamWaitEvent(stream, s->a_in[slot], 0));
    RT_CHECK(s, cudaStreamWaitEvent(stream, s->a_done[slot], 0));
    /* ... and after the count kernel of two ticks ago, whose input this kernel clears */
    RT_CHECK(s, cudaStreamWaitEvent(stream, s->a_cnt[(slot + 1) % PVE_ASYNC_SLOTS], 0));
    rc = launch_step(s, s->a_act[slot], *out_dev, stream);
    if (rc != PVE_OK) return rc;
    s->next_total = -1;
    RT_CHECK(s, cudaEventRecord(s->a_k[slot], stream));
    /* the NEXT tick's row count goes home behind the kernel, on its own stream */
    RT_CHECK(s, cudaStreamWaitEvent(s->s_cnt, s->a_k[slot], 0));
    pve_total_kernel<<<1, 32, 0, s->s_cnt>>>(s->st.gs_read, s->n_groups, s->a_total + slot);
    RT_CHECK(s, cudaGetLastError());
    RT_CHECK(s, cudaEventRecord(s->a_cnt[slot], s->s_cnt));
    s->a_rows[slot] = A;
    s->a_odev[slot] = *out_dev; s->a_ohost[slot] = *out_host; s->a_mask[slot] = copy_mask;
    s->a_seq += 1;
    /* the copy-out of the tick before this one: its row count arrived a whole tick ago, so nothing blocks here and
     * the GPU already has this tick's kernel queued */
    if (s->a_copied < s->a_seq - 1) {
        rc = async_copy_out(s, s->a_seq - 2);
        if (rc != PVE_OK) return rc;
    }
    return PVE_OK;
#endif
}

int64_t pve_host_wait(pve_scene *s) {
    if (!s) return PVE_EINVAL;
#ifdef PVE_HOST_EMULATION
    return PVE_ESTATE;
#else
    if (s->a_seq <= s->a_waited) { snprintf(s->err, sizeof s->err, "no tick in flight"); return PVE_ESTATE; }
    while (s->a_copied <= s->a_waited) {                                      /* the newest tick: enqueue its copy-out now */
        int32_t rc = async_copy_out(s, s->a_copied);
        if (rc != PVE_OK) return rc;
    }
    const int slot = (int)(s->a_waited % PVE_ASYNC_SLOTS);                    /* the oldest one */
    RT_CHECK(s, cudaEventSynchronize(s->a_done[slot]));
    s->a_waited += 1;
    return s->a_rows[slot];
#endif
}

int32_t pve_set_state(pve_scene *s, const pve_state_view *in, void *stream_) {
    if (!s || !in) return PVE_EINVAL;
    pve_stream_t stream = (pve_stream_t)stream_;
    const int B = s->cfg.n_envs;
    const size_t nv = (size_t)B * s->cfg.veh_cap;
    RT_CHECK(s, rt_copy(s->st.hdr, in->hdr, sizeof(pve_env_header) * (size_t)B, stream));
    RT_CHECK(s, rt_copy(s->st.p, in->p, sizeof(double) * nv, stream));
    RT_CHECK(s, rt_copy(s->st.v, in->v, sizeof(double) * nv, stream));
    RT_CHECK(s, rt_copy(s->st.a, in->a, sizeof(double) * nv, stream));
    RT_CHECK(s, rt_copy(s->st.js, in->jerk_sum, sizeof(double) * nv, stream));
    RT_CHECK(s, rt_copy(s->st.meta, in->meta, sizeof(pve_veh_meta) * nv, stream));
    RT_CHECK(s, rt_copy(s->st.row0[s->phase], in->row0, sizeof(float) * nv * PVE_OBS_W, stream));
#ifndef PVE_HOST_EMULATION
    if (s->poisson) pve_recount_kernel<true><<<(B + 127) / 128, 128, 0, stream>>>(s->st, s->poi, B, s->cfg.veh_cap, 0);
    else pve_recount_kernel<false><<<(B + 127) / 128, 128, 0, stream>>>(s->st, s->spawn_tick, B, s->cfg.veh_cap, s->prm.K);
    RT_CHECK(s, cudaGetLastError());
#else
    if (s->poisson) emul_recount<true>(s->st, s->poi, B, s->cfg.veh_cap, 0);
    else emul_recount<false>(s->st, s->spawn_tick, B, s->cfg.veh_cap, s->prm.K);
#endif
    s->next_total = -1;
    s->order_age = -1;
    return launch_gsum(s, stream);
}

int32_t pve_get_state(pve_scene *s, const pve_state_view *out, void *stream_) {
    if (!s || !out) return PVE_EINVAL;
    pve_stream_t stream = (pve_stream_t)stream_;
    const int B = s->cfg.n_envs;
    const size_t nv = (size_t)B * s->cfg.veh_cap;
    RT_CHECK(s, rt_copy(out->hdr, s->st.hdr, sizeof(pve_env_header) * (size_t)B, stream));
    RT_CHECK(s, rt_copy(out->p, s->st.p, sizeof(double) * nv, stream));
    RT_CHECK(s, rt_copy(out->v, s->st.v, sizeof(double) * nv, stream));
    RT_CHECK(s, rt_copy(out->a, s->st.a, sizeof(double) * nv, stream));
    RT_CHECK(s, rt_copy(out->jerk_sum, s->st.js, sizeof(double) * nv, stream));
    RT_CHECK(s, rt_copy(out->meta, s->st.meta, sizeof(pve_veh_meta) * nv, stream));
    RT_CHECK(s, rt_copy(out->row0, s->st.row0[s->phase], sizeof(float) * nv * PVE_OBS_W, stream));
    RT_CHECK(s, rt_sync(stream));
    return PVE_OK;
}

const float *pve_row0_dev(const pve_scene *s) { return s ? s->st.row0[s->phase] : nullptr; }
const float *pve_row0_prev_dev(const pve_scene *s) { return s ? s->st.row0[s->phase ^ 1] : nullptr; }
const pve_veh_meta *pve_meta_dev(const pve_scene *s) { return s ? s->st.meta : nullptr; }
const pve_env_header *pve_hdr_dev(const pve_scene *s) { return s ? s->st.hdr : nullptr; }
const double *pve_env_stats_dev(const pve_scene *s) { return s ? s->st.stats : nullptr; }
static_assert(PVE_ENV_NSTAT == PVE_NSTAT, "per-intersection statistics");
int64_t pve_smem_bytes(const pve_scene *s) { return s ? (int64_t)s->smem_bytes : 0; }
int32_t pve_threads(const pve_scene *s) { return s ? s->threads : 0; }
int32_t pve_launch_info(const pve_scene *s, int32_t out[8]) {
    if (!s || !out) return PVE_EINVAL;
    for (int i = 0; i < 8; ++i) out[i] = 0;
#ifndef PVE_HOST_EMULATION
    if (s->dual) {
        out[0] = 1; out[1] = PVE_SMALL_VC; out[2] = PVE_SMALL_AC; out[3] = PVE_SMALL_NT;
        out[4] = (int32_t)PveLayout<PVE_SMALL_VC, PVE_SMALL_AC>::BYTES;
    }
#endif
    return PVE_OK;
}
#ifdef PVE_PHASE_TIMING
const void *pve_debug_stamps(const pve_scene *s) { return s ? s->st.dbg : nullptr; }
#endif
int32_t pve_veh_cap(const pve_scene *s) { return s ? s->cfg.veh_cap : 0; }
int32_t pve_agent_cap(const pve_scene *s) { return s ? s->cfg.agent_cap : 0; }

int32_t pve_stats(pve_scene *s, pve_counters *out_dev, void *stream_) {
    if (!s || !out_dev) return PVE_EINVAL;
    pve_stream_t stream = (pve_stream_t)stream_;
#ifndef PVE_HOST_EMULATION
    pve_stats_kernel<<<1, 256, 0, stream>>>(s->st, s->cfg.n_envs, s->counters_dev);
    RT_CHECK(s, cudaGetLastError());
#else
    emul_stats(s->st, s->cfg.n_envs, s->counters_dev);
#endif
    RT_CHECK(s, rt_copy(out_dev, s->counters_dev, sizeof(double) * 16, stream));
    return PVE_OK;
}

/* ---- factored observation -> obs ------------------------------------------------------------ */
int64_t pve_expand_obs_host(const int32_t *off, int32_t b0, int32_t b1, int64_t out_cap, const float *r0,
                            const float *pr, const int16_t *src, float *obs) {
    if (!off || !r0 || !pr || !src || !obs || b0 < 0 || b1 < b0) return PVE_EINVAL;
    const size_t row_bytes = sizeof(float) * PVE_OBS_W;
    int64_t bad = 0;
    for (int32_t b = b0; b < b1; ++b) {
        const int64_t o0 = off[b], o1 = off[b + 1];
        if (o0 < 0 || o1 < o0) { ++bad; continue; }
        if (o1 > out_cap) continue;                             /* rows the step did not write */
        for (int64_t r = o0; r < o1; ++r) {
            float *dst = obs + (size_t)r * PVE_OBS_H * PVE_OBS_W;
            for (int q = 0; q < PVE_OBS_H; ++q) {
                int64_t idx = 0;
                const int k = pve_obs_src_decode(src[(size_t)r * 8 + q], o1 - o0, &idx);
                float *d = dst + q * PVE_OBS_W;
                if (k > 0) memcpy(d, (k == 1 ? r0 : pr) + (size_t)(o0 + idx) * PVE_OBS_W, row_bytes);
                else if (k == 0) memset(d, 0, row_bytes);
                else {
                    ++bad;
                    const uint32_t w = PVE_NAN_BITS;
                    for (int i = 0; i < PVE_OBS_W; ++i) memcpy(d + i, &w, sizeof w);
                }
            }
        }
    }
    return bad;
}

int32_t pve_expand_obs(const int32_t *off_dev, int32_t B, int64_t out_cap, const float *r0_dev, const float *pr_dev,
                       const int16_t *src_dev, float *obs_dev, void *stream) {
    if (!off_dev || !r0_dev || !pr_dev || !src_dev || !obs_dev || B < 0) return PVE_EINVAL;
    if (B == 0) return PVE_OK;
#ifndef PVE_HOST_EMULATION
    pve_expand_obs_kernel<<<B, 128, 0, (pve_stream_t)stream>>>(off_dev, out_cap, (const pve_v4 *)r0_dev, (const pve_v4 *)pr_dev,
                                                               src_dev, (pve_v4 *)obs_dev);
    return cudaGetLastError() == cudaSuccess ? PVE_OK : PVE_ECUDA;
#else
    (void)stream;
    return pve_expand_obs_host(off_dev, 0, B, out_cap, r0_dev, pr_dev, src_dev, obs_dev) >= 0 ? PVE_OK : PVE_EINVAL;
#endif
}

/* ---- actor (N1) ---------------------------------------------------------------------------- */
struct pve_actor {
    float *w_dev;                /* flat fp32 parameters (FFMA kernel) */
    uint32_t *pw_dev;            /* split bf16 fragments + vectors (tensor-core kernel) */
    int *ticket;                 /* [2] work counter + exit counter of the kernel, zero between launches */
    int device;
    int blocks_ffma, blocks_mma; /* one resident wave of CTAs each */
    int use_mma;                 /* 3 = by size (default: tcgen05 from PVE_TC_MIN_ROWS candidate rows on, mma.sync below: its fixed cost is
                                  * ~4 us lower), 2 = tcgen05 kernel (PVE_ACTOR_IMPL=tc5), 1 = mma.sync kernel (=mma), 0 = CUDA cores (=ffma) */
    uint16_t *tw_dev;            /* shared-memory image of the split weights (tcgen05 kernel) */
    PvtVecs vecs;                /* bias / LayerNorm / last-layer vectors: a kernel parameter of the tcgen05 kernel */
    int blocks_tc;
    float *zero_dev;             /* [28] zeros + [1] the action of an all-zero row (a missing neighbour, TIS:1334) */
};

#define PVE_TC_MIN_ROWS 16384     /* candidate rows (vehicle slots / matrix rows) from which the tcgen05 kernels are the faster ones */
#ifndef PVE_HOST_EMULATION
static cudaError_t launch_actor(pve_actor *a, const float *rows, const pve_veh_meta *meta, const int32_t *n_veh,
                                const float *noise, float noise_scale, float *actions, int slots_per_env, int n_env,
                                long long n_slots, pve_stream_t stream, const int32_t *limit_dev = nullptr, int limit_mult = 1,
                                const uint8_t *mask = nullptr, int slot_step = 1);
#endif

int32_t pve_actor_create(const float *weights_host, int32_t n_floats, int32_t device, pve_actor **out) {
    if (!weights_host || !out || n_floats != PVE_ACTOR_FLOATS) return PVE_EINVAL;
#ifdef PVE_HOST_EMULATION
    (void)device;
    return PVE_ESTATE;                       /* device only */
#else
    if (cudaSetDevice(device) != cudaSuccess) return PVE_ECUDA;
    pve_actor *a = (pve_actor *)calloc(1, sizeof(pve_actor));
    if (!a) return PVE_ENOMEM;
    a->device = device;
    a->use_mma = 3;
    if (const char *impl = getenv("PVE_ACTOR_IMPL")) a->use_mma = strcmp(impl, "ffma") == 0 ? 0 : strcmp(impl, "mma") == 0 ? 1 : strcmp(impl, "tc5") == 0 ? 2 : 3;
    int sms = 0, per_sm = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || sms <= 0) sms = 148;
    bool ok = cudaFuncSetAttribute(pve_actor_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PVA_SMEM_BYTES) == cudaSuccess
              && cudaFuncSetAttribute(pve_actor_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PVM_SMEM_BYTES) == cudaSuccess
              && cudaFuncSetAttribute(pve_actor_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PVT_ACTOR_SMEM) == cudaSuccess;
    if (ok) {
        a->blocks_tc = sms;                  /* one persistent CTA per SM (three groups of 128 rows + the producer warp) */
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pve_actor_kernel, PVA_THREADS, PVA_SMEM_BYTES) != cudaSuccess || per_sm < 1) per_sm = 1;
        a->blocks_ffma = per_sm * sms;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pve_actor_mma_kernel, PVM_THREADS, PVM_SMEM_BYTES) != cudaSuccess || per_sm < 1) per_sm = 1;
        a->blocks_mma = per_sm * sms;
    }
    uint32_t *packed = ok ? (uint32_t *)malloc(sizeof(uint32_t) * PVM_WORDS) : nullptr;
    ok = ok && packed;
    if (ok) pvm_pack(weights_host, packed);
    uint16_t *image = ok ? (uint16_t *)malloc(PVT_W_BYTES) : nullptr;
    ok = ok && image;
    if (ok) {
        pvt_pack(weights_host + PVA_W1, weights_host + PVA_B1, weights_host + PVA_W2, weights_host + PVA_B2, 0, image);
        pvt_vecs_actor(weights_host, &a->vecs);
    }
    ok = ok && cudaMalloc((void **)&a->tw_dev, PVT_W_BYTES) == cudaSuccess
            && cudaMemcpy(a->tw_dev, image, PVT_W_BYTES, cudaMemcpyHostToDevice) == cudaSuccess;
    free(image);
    ok = ok && cudaMalloc((void **)&a->w_dev, sizeof(float) * PVE_ACTOR_FLOATS) == cudaSuccess
            && cudaMalloc((void **)&a->pw_dev, sizeof(uint32_t) * PVM_WORDS) == cudaSuccess
            && cudaMalloc((void **)&a->ticket, 2 * sizeof(int)) == cudaSuccess
            && cudaMemcpy(a->w_dev, weights_host, sizeof(float) * PVE_ACTOR_FLOATS, cudaMemcpyHostToDevice) == cudaSuccess
            && cudaMemcpy(a->pw_dev, packed, sizeof(uint32_t) * PVM_WORDS, cudaMemcpyHostToDevice) == cudaSuccess
            && cudaMemset(a->ticket, 0, 2 * sizeof(int)) == cudaSuccess;
    free(packed);
    /* the action of the all-zero row of a missing neighbour (TIS:1334), once per network and finished before the handle
     * is handed out, so that pushes on any stream may read it (the weights of a handle never change) */
    ok = ok && cudaMalloc((void **)&a->zero_dev, 32 * sizeof(float)) == cudaSuccess
            && cudaMemset(a->zero_dev, 0, 32 * sizeof(float)) == cudaSuccess
            && launch_actor(a, a->zero_dev, nullptr, nullptr, nullptr, 0.f, a->zero_dev + 28, PVA_TILE, 1, 1, nullptr,
                            nullptr, 1, nullptr, 1) == cudaSuccess
            && cudaDeviceSynchronize() == cudaSuccess;
    if (!ok) {
        fprintf(stderr, "pve_actor_create: %s\n", cudaGetErrorString(cudaPeekAtLastError()));
        cudaFree(a->w_dev); cudaFree(a->pw_dev); cudaFree(a->tw_dev); cudaFree(a->ticket); cudaFree(a->zero_dev); free(a);
        cudaGetLastError();
        return PVE_ECUDA;
    }
    *out = a;
    return PVE_OK;
#endif
}

void pve_actor_destroy(pve_actor *a) {
    if (!a) return;
#ifndef PVE_HOST_EMULATION
    cudaFree(a->w_dev);
    cudaFree(a->pw_dev);
    cudaFree(a->tw_dev);
    cudaFree(a->ticket);
    cudaFree(a->zero_dev);
#endif
    free(a);
}

#ifndef PVE_HOST_EMULATION
static cudaError_t launch_actor(pve_actor *a, const float *rows, const pve_veh_meta *meta, const int32_t *n_veh,
                                const float *noise, float noise_scale, float *actions, int slots_per_env, int n_env,
                                long long n_slots, pve_stream_t stream, const int32_t *limit_dev, int limit_mult,
                                const uint8_t *mask, int slot_step) {
    const int impl = a->use_mma == 3 ? (n_slots >= PVE_TC_MIN_ROWS ? 2 : 1) : a->use_mma;
    if (impl == 2) {
        const int blocks = n_env < a->blocks_tc ? n_env : a->blocks_tc;
        pve_actor_tc_kernel<<<blocks, PVT_THREADS_ACTOR, PVT_ACTOR_SMEM, stream>>>(a->vecs, a->tw_dev, rows, meta, n_veh, noise, noise_scale,
                                                                                actions, slots_per_env, n_env, n_slots, a->ticket, limit_dev, limit_mult, mask, slot_step);
    } else if (impl) {
        const int blocks = n_env < a->blocks_mma ? n_env : a->blocks_mma;
        pve_actor_mma_kernel<<<blocks, PVM_THREADS, PVM_SMEM_BYTES, stream>>>(a->pw_dev, rows, meta, n_veh, noise, noise_scale,
                                                                           actions, slots_per_env, n_env, n_slots, a->ticket, limit_dev, limit_mult, mask, slot_step);
    } else {
        const int blocks = n_env < a->blocks_ffma ? n_env : a->blocks_ffma;
        pve_actor_kernel<<<blocks, PVA_THREADS, PVA_SMEM_BYTES, stream>>>(a->w_dev, rows, meta, n_veh, noise, noise_scale,
                                                                       actions, slots_per_env, n_env, n_slots, a->ticket, limit_dev, limit_mult, mask, slot_step);
    }
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) fprintf(stderr, "pve actor launch: %s\n", cudaGetErrorString(e));
    return e;
}
#endif

#if defined(PVT_X_TRACE) && !defined(PVE_HOST_EMULATION)
extern "C" int32_t pve_debug_trace(long long *out, int32_t n) {          /* experiment builds only */
    return cudaMemcpyFromSymbol(out, pvt_trace_buf, sizeof(long long) * n) == cudaSuccess ? 0 : -1;
}
#endif

int32_t pve_actor_forward(pve_actor *a, const float *rows_dev, int64_t n_rows, float *actions_dev, void *stream_) {
    if (!a || !rows_dev || !actions_dev || n_rows < 0) return PVE_EINVAL;
#ifdef PVE_HOST_EMULATION
    (void)stream_;
    return PVE_ESTATE;
#else
    if (n_rows == 0) return PVE_OK;
    if (n_rows > 0x7fffffffLL) return PVE_EINVAL;             /* slot indices are queued as 32-bit */
    const long long groups = (n_rows + PVA_TILE - 1) / PVA_TILE;             /* "intersections" of 128 rows */
    return launch_actor(a, rows_dev, nullptr, nullptr, nullptr, 0.f, actions_dev, PVA_TILE, (int)groups, (long long)n_rows,
                        (pve_stream_t)stream_) == cudaSuccess ? PVE_OK : PVE_ECUDA;
#endif
}

int32_t pve_act(pve_scene *s, pve_actor *a, const float *noise_dev, float noise_scale, float *actions_dev,
                void *stream_) {
    if (!s || !a || !actions_dev) return PVE_EINVAL;
#ifdef PVE_HOST_EMULATION
    (void)noise_dev; (void)noise_scale; (void)stream_;
    snprintf(s->err, sizeof(s->err), "pve_act: the actor kernel exists on the device only");
    return PVE_ESTATE;
#else
    if (a->device != s->device) {
        snprintf(s->err, sizeof(s->err), "pve_act: actor lives on device %d, scene on %d", a->device, s->device);
        return PVE_EINVAL;
    }
    const int B = s->cfg.n_envs, VCc = s->prm.VC;
    RT_CHECK(s, launch_actor(a, pve_row0_dev(s), s->st.meta, s->st.n_veh, noise_dev, noise_scale, actions_dev, VCc, B,
                             (long long)B * (long long)VCc, (pve_stream_t)stream_));
    return PVE_OK;
#endif
}

int32_t pve_rollout(pve_scene *s, pve_actor *a, int32_t n_ticks, const float *noise_dev, float noise_scale,
                    float *actions_dev, const pve_outputs *out, void *stream) {
    if (!s || !a || !actions_dev || !out || n_ticks < 0) return PVE_EINVAL;
    for (int32_t t = 0; t < n_ticks; ++t) {
        int32_t rc = pve_act(s, a, noise_dev, noise_scale, actions_dev, stream);
        if (rc != PVE_OK) return rc;
        rc = pve_step(s, actions_dev, out, stream);
        if (rc != PVE_OK) return rc;
    }
    return PVE_OK;
}

int32_t pve_actor_forward_n(pve_actor *a, const float *rows_dev, int64_t max_rows, const int32_t *n_rows_dev,
                            int32_t mult, float *actions_dev, void *stream_) {
    if (!a || !rows_dev || !actions_dev || !n_rows_dev || max_rows < 0 || mult < 1) return PVE_EINVAL;
#ifdef PVE_HOST_EMULATION
    (void)stream_;
    return PVE_ESTATE;
#else
    if (max_rows == 0) return PVE_OK;
    if (max_rows > 0x7fffffffLL) return PVE_EINVAL;
    const long long groups = (max_rows + PVA_TILE - 1) / PVA_TILE;
    return launch_actor(a, rows_dev, nullptr, nullptr, nullptr, 0.f, actions_dev, PVA_TILE, (int)groups, (long long)max_rows,
                        (pve_stream_t)stream_, n_rows_dev, mult) == cudaSuccess ? PVE_OK : PVE_ECUDA;
#endif
}

/* ---- critic + n-step folding + replay writer (N2) ------------------------------------------ */
struct pve_critic {
    float *w_dev;                /* flat fp32 parameters (FFMA kernel) */
    uint32_t *pw_dev;            /* split bf16 fragments + vectors (tensor-core kernel) */
    int device, blocks, blocks_mma;
    int use_mma;                 /* 3 = by size (default), 2 = tcgen05 kernel (PVE_CRITIC_IMPL=tc5), 1 = mma.sync kernel (=mma), 0 = CUDA cores (=ffma) */
    uint16_t *tw_dev;            /* shared-memory image of the split weights (tcgen05 kernel) */
    PvtVecs vecs;
    int blocks_tc;
};

int32_t pve_critic_create(const float *weights_host, int32_t n_floats, int32_t device, pve_critic **out) {
    if (!weights_host || !out || n_floats != PVE_CRITIC_FLOATS) return PVE_EINVAL;
#ifdef PVE_HOST_EMULATION
    (void)device;
    return PVE_ESTATE;                       /* device only */
#else
    if (cudaSetDevice(device) != cudaSuccess) return PVE_ECUDA;
    pve_critic *c = (pve_critic *)calloc(1, sizeof(pve_critic));
    if (!c) return PVE_ENOMEM;
    c->device = device;
    int sms = 0, per_sm = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || sms <= 0) sms = 148;
    c->use_mma = 3;
    if (const char *impl = getenv("PVE_CRITIC_IMPL")) c->use_mma = strcmp(impl, "ffma") == 0 ? 0 : strcmp(impl, "mma") == 0 ? 1 : strcmp(impl, "tc5") == 0 ? 2 : 3;
    /* both row-0 strides: observation blocks (pve_critic_forward) and the factored log's rows (pve_nstep_push_factored) */
    bool ok = cudaFuncSetAttribute(pve_critic_kernel<PVN_OBS>, cudaFuncAttributeMaxDynamicSharedMemorySize, PVC_SMEM_BYTES) == cudaSuccess
              && cudaFuncSetAttribute(pve_critic_mma_kernel<PVN_OBS>, cudaFuncAttributeMaxDynamicSharedMemorySize, PVQ_SMEM_BYTES) == cudaSuccess
              && cudaFuncSetAttribute(pve_critic_tc_kernel<PVN_OBS>, cudaFuncAttributeMaxDynamicSharedMemorySize, PVT_CRITIC_SMEM) == cudaSuccess
              && cudaFuncSetAttribute(pve_critic_kernel<PVE_OBS_W>, cudaFuncAttributeMaxDynamicSharedMemorySize, PVC_SMEM_BYTES) == cudaSuccess
              && cudaFuncSetAttribute(pve_critic_mma_kernel<PVE_OBS_W>, cudaFuncAttributeMaxDynamicSharedMemorySize, PVQ_SMEM_BYTES) == cudaSuccess
              && cudaFuncSetAttribute(pve_critic_tc_kernel<PVE_OBS_W>, cudaFuncAttributeMaxDynamicSharedMemorySize, PVT_CRITIC_SMEM) == cudaSuccess;
    c->blocks_tc = sms;                      /* one persistent CTA per SM */
    if (ok && (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pve_critic_kernel<PVN_OBS>, PVC_THREADS, PVC_SMEM_BYTES) != cudaSuccess || per_sm < 1)) per_sm = 1;
    c->blocks = per_sm * sms;
    if (ok && (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pve_critic_mma_kernel<PVN_OBS>, PVQ_THREADS, PVQ_SMEM_BYTES) != cudaSuccess || per_sm < 1)) per_sm = 1;
    c->blocks_mma = per_sm * sms;
    uint32_t *packed = ok ? (uint32_t *)malloc(sizeof(uint32_t) * PVQ_WORDS) : nullptr;
    ok = ok && packed;
    if (ok) pvq_pack(weights_host, packed);
    uint16_t *image = ok ? (uint16_t *)malloc(PVT_W_BYTES) : nullptr;
    ok = ok && image;
    if (ok) {
        pvt_pack(weights_host + PVC_W1, weights_host + PVC_B1, weights_host + PVC_W2, weights_host + PVC_B2, 1, image);
        pvt_vecs_critic(weights_host, &c->vecs);
    }
    ok = ok && cudaMalloc((void **)&c->tw_dev, PVT_W_BYTES) == cudaSuccess
            && cudaMemcpy(c->tw_dev, image, PVT_W_BYTES, cudaMemcpyHostToDevice) == cudaSuccess;
    free(image);
    ok = ok && cudaMalloc((void **)&c->w_dev, sizeof(float) * PVE_CRITIC_FLOATS) == cudaSuccess
            && cudaMalloc((void **)&c->pw_dev, sizeof(uint32_t) * PVQ_WORDS) == cudaSuccess
            && cudaMemcpy(c->w_dev, weights_host, sizeof(float) * PVE_CRITIC_FLOATS, cudaMemcpyHostToDevice) == cudaSuccess
            && cudaMemcpy(c->pw_dev, packed, sizeof(uint32_t) * PVQ_WORDS, cudaMemcpyHostToDevice) == cudaSuccess;
    free(packed);
    if (!ok) { fprintf(stderr, "pve_critic_create: %s\n", cudaGetErrorString(cudaPeekAtLastError())); cudaFree(c->w_dev); cudaFree(c->pw_dev); cudaFree(c->tw_dev); free(c); cudaGetLastError(); return PVE_ECUDA; }
    *out = c;
    return PVE_OK;
#endif
}

void pve_critic_destroy(pve_critic *c) {
    if (!c) return;
#ifndef PVE_HOST_EMULATION
    cudaFree(c->w_dev);
    cudaFree(c->pw_dev);
    cudaFree(c->tw_dev);
#endif
    free(c);
}

#ifndef PVE_HOST_EMULATION
}  /* extern "C" */
/* q_dev[i] = Q(obs_dev + i * STRIDE, act7_dev[i]) for i < min(max_rows, n_rows_dev[0]) */
template <int STRIDE>
static int32_t critic_forward(pve_critic *c, const float *obs_dev, const float *act7_dev, int64_t max_rows,
                              const int32_t *n_rows_dev, float *q_dev, pve_stream_t stream) {
    if (max_rows == 0) return PVE_OK;
    const long long tiles = (max_rows + PVC_TILE - 1) / PVC_TILE;              /* both kernels: 128 agents per tile */
    const int impl = c->use_mma == 3 ? (max_rows >= PVE_TC_MIN_ROWS ? 2 : 1) : c->use_mma;
    if (impl == 2) {
        const long long ctas = (tiles + PVT_GROUPS - 1) / PVT_GROUPS;
        const int blocks = (int)(ctas < c->blocks_tc ? ctas : c->blocks_tc);
        pve_critic_tc_kernel<STRIDE><<<blocks, PVT_THREADS_CRITIC, PVT_CRITIC_SMEM, stream>>>(c->vecs, c->tw_dev, obs_dev, act7_dev, q_dev,
                                                                                           (long long)max_rows, n_rows_dev);
    } else if (impl) {
        const int blocks = (int)(tiles < c->blocks_mma ? tiles : c->blocks_mma);
        pve_critic_mma_kernel<STRIDE><<<blocks, PVQ_THREADS, PVQ_SMEM_BYTES, stream>>>(c->pw_dev, obs_dev, act7_dev, q_dev,
                                                                                      (long long)max_rows, n_rows_dev);
    } else {
        const int blocks = (int)(tiles < c->blocks ? tiles : c->blocks);
        pve_critic_kernel<STRIDE><<<blocks, PVC_THREADS, PVC_SMEM_BYTES, stream>>>(c->w_dev, obs_dev, act7_dev, q_dev,
                                                                                  (long long)max_rows, n_rows_dev);
    }
    return cudaGetLastError() == cudaSuccess ? PVE_OK : PVE_ECUDA;
}
extern "C" {
#endif

int32_t pve_critic_forward(pve_critic *c, const float *obs_dev, const float *act7_dev, int64_t max_rows,
                           const int32_t *n_rows_dev, float *q_dev, void *stream_) {
    if (!c || !obs_dev || !act7_dev || !q_dev || max_rows < 0) return PVE_EINVAL;
#ifdef PVE_HOST_EMULATION
    (void)n_rows_dev; (void)stream_;
    return PVE_ESTATE;
#else
    return critic_forward<PVN_OBS>(c, obs_dev, act7_dev, max_rows, n_rows_dev, q_dev, (pve_stream_t)stream_);
#endif
}

struct pve_nstep {
    PvnTable T;
    PvnReplay R;
    float *act7, *q;             /* [out_cap][7], [out_cap] target actions and bootstrap values of the last push */
    uint32_t *plan;              /* [out_cap] */
    int32_t *blk_count;          /* [n_blk] */
    long long *blk_base;         /* [n_blk] */
    long long *counters;         /* [4] device */
    long long out_cap, pushes;
    int n_blk, device, fold_blocks;
    /* pve_nstep_push_scene (allocated on first use): referenced-row marks and actions of last tick's stored rows,
     * [B][veh_cap]; a factored folder: the same for the referenced prev_row0 rows, [out_cap] */
    uint8_t *need;
    float *mu_prev;
    size_t scene_slots;
    PvnFactored F;               /* the factored frame log (pve_nstep_create_factored; T.log is null then) */
    float *mu0;                  /* factored: [out_cap] the target actor on this tick's row0_out */
    char err[256];
#ifndef PVE_HOST_EMULATION
    cudaEvent_t fold_ev[2];      /* pve_nstep_set_profiling: around the fold kernel of the last push */
#endif
    int profiling;
};

static int32_t nstep_refuse(pve_nstep *f, const char *msg) {
    snprintf(f->err, sizeof f->err, "%s", msg);
    return PVE_EINVAL;
}

void pve_nstep_destroy(pve_nstep *f) {
    if (!f) return;
#ifndef PVE_HOST_EMULATION
    cudaFree(f->T.key); cudaFree(f->T.fill); cudaFree(f->T.rew); cudaFree(f->T.fidx); cudaFree(f->T.log);
    cudaFree(f->R.state); cudaFree(f->R.action); cudaFree(f->R.reward); cudaFree(f->R.next_state); cudaFree(f->R.done);
    cudaFree(f->need); cudaFree(f->mu_prev); cudaFree(f->mu0);
    cudaFree(f->F.row0); cudaFree(f->F.prev); cudaFree(f->F.src); cudaFree(f->F.off);
    if (f->profiling) { cudaEventDestroy(f->fold_ev[0]); cudaEventDestroy(f->fold_ev[1]); }
    cudaFree(f->act7); cudaFree(f->q); cudaFree(f->plan); cudaFree(f->blk_count); cudaFree(f->blk_base); cudaFree(f->counters);
#endif
    free(f);
}

static int32_t nstep_create(int32_t n_envs, int32_t uid_slots, int32_t seq_max_step, int64_t out_cap,
                            int64_t buffer_size, int32_t device, bool factored, pve_nstep **out) {
    if (!out || n_envs < 1 || uid_slots < 16 || (uid_slots & (uid_slots - 1)) != 0 || seq_max_step < 0
        || seq_max_step + 2 > PVN_MAX_M || out_cap < 1 || buffer_size - 1 < out_cap)
        return PVE_EINVAL;
#ifdef PVE_HOST_EMULATION
    (void)device; (void)factored;
    return PVE_ESTATE;                       /* device only */
#else
    if (cudaSetDevice(device) != cudaSuccess) return PVE_ECUDA;
    pve_nstep *f = (pve_nstep *)calloc(1, sizeof(pve_nstep));
    if (!f) return PVE_ENOMEM;
    f->device = device;
    f->out_cap = out_cap;
    f->T.B = n_envs; f->T.U = uid_slots; f->T.S = seq_max_step; f->T.M = seq_max_step + 2; f->T.out_cap = out_cap;
    if ((long long)f->T.M * out_cap > 0x7fffffffLL) { free(f); return PVE_EINVAL; }   /* frame references are 32-bit log rows */
    f->R.cap = buffer_size - 1;
    f->n_blk = (int)((out_cap + PVN_PLAN_THREADS - 1) / PVN_PLAN_THREADS);
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || sms <= 0) sms = 148;
    f->fold_blocks = sms * 8;
    const size_t slots = (size_t)n_envs * uid_slots, cap = (size_t)f->R.cap, oc = (size_t)out_cap;
    bool ok = cudaMalloc((void **)&f->T.key, slots * 8) == cudaSuccess
              && cudaMalloc((void **)&f->T.fill, slots * 2) == cudaSuccess
              && cudaMalloc((void **)&f->T.rew, slots * f->T.M * sizeof(float)) == cudaSuccess
              && cudaMalloc((void **)&f->T.fidx, slots * f->T.M * sizeof(int32_t)) == cudaSuccess
              && (factored || cudaMalloc((void **)&f->T.log, (size_t)f->T.M * oc * PVN_OBS * sizeof(float)) == cudaSuccess)
              && (!factored || (cudaMalloc((void **)&f->F.row0, (size_t)f->T.M * oc * PVE_OBS_W * sizeof(float)) == cudaSuccess
                                && cudaMalloc((void **)&f->F.prev, (size_t)f->T.M * oc * PVE_OBS_W * sizeof(float)) == cudaSuccess
                                && cudaMalloc((void **)&f->F.src, (size_t)f->T.M * oc * 8 * sizeof(int16_t)) == cudaSuccess
                                && cudaMalloc((void **)&f->F.off, (size_t)f->T.M * (n_envs + 1) * sizeof(int32_t)) == cudaSuccess
                                && cudaMalloc((void **)&f->need, oc) == cudaSuccess
                                && cudaMalloc((void **)&f->mu_prev, oc * sizeof(float)) == cudaSuccess
                                && cudaMalloc((void **)&f->mu0, oc * sizeof(float)) == cudaSuccess))
              && cudaMalloc((void **)&f->R.state, cap * PVN_OBS * sizeof(float)) == cudaSuccess
              && cudaMalloc((void **)&f->R.next_state, cap * PVN_OBS * sizeof(float)) == cudaSuccess
              && cudaMalloc((void **)&f->R.action, cap * PVE_OBS_H * sizeof(float)) == cudaSuccess
              && cudaMalloc((void **)&f->R.reward, cap * sizeof(float)) == cudaSuccess
              && cudaMalloc((void **)&f->R.done, cap) == cudaSuccess
              && cudaMalloc((void **)&f->act7, oc * PVE_OBS_H * sizeof(float)) == cudaSuccess
              && cudaMalloc((void **)&f->q, oc * sizeof(float)) == cudaSuccess
              && cudaMalloc((void **)&f->plan, oc * sizeof(uint32_t)) == cudaSuccess
              && cudaMalloc((void **)&f->blk_count, (size_t)f->n_blk * sizeof(int32_t)) == cudaSuccess
              && cudaMalloc((void **)&f->blk_base, (size_t)f->n_blk * sizeof(long long)) == cudaSuccess
              && cudaMalloc((void **)&f->counters, 4 * sizeof(long long)) == cudaSuccess;
    ok = ok && cudaMemset(f->T.key, 0xFF, slots * 8) == cudaSuccess && cudaMemset(f->T.fill, 0, slots * 2) == cudaSuccess
            && cudaMemset(f->counters, 0, 4 * sizeof(long long)) == cudaSuccess
            && cudaMemset(f->q, 0, oc * sizeof(float)) == cudaSuccess && cudaMemset(f->R.done, 0, cap) == cudaSuccess
            && cudaMemset(f->R.reward, 0, cap * sizeof(float)) == cudaSuccess;
    if (!ok) { cudaGetLastError(); pve_nstep_destroy(f); return PVE_ENOMEM; }
    *out = f;
    return PVE_OK;
#endif
}

int32_t pve_nstep_create(int32_t n_envs, int32_t uid_slots, int32_t seq_max_step, int64_t out_cap,
                         int64_t buffer_size, int32_t device, pve_nstep **out) {
    return nstep_create(n_envs, uid_slots, seq_max_step, out_cap, buffer_size, device, false, out);
}

int32_t pve_nstep_create_factored(int32_t n_envs, int32_t uid_slots, int32_t seq_max_step, int64_t out_cap,
                                  int64_t buffer_size, int32_t device, pve_nstep **out) {
    return nstep_create(n_envs, uid_slots, seq_max_step, out_cap, buffer_size, device, true, out);
}

#ifndef PVE_HOST_EMULATION
static int32_t nstep_fold(pve_nstep *f, const pve_outputs *O, double gamma, pve_critic *target_critic, void *stream_);
#endif

int32_t pve_nstep_push(pve_nstep *f, const pve_outputs *O, double gamma, pve_actor *target_actor,
                       pve_critic *target_critic, void *stream_) {
    if (f && f->F.row0) return nstep_refuse(f, "pve_nstep_push: this folder keeps a factored frame log, push with pve_nstep_push_factored");
    if (!f || !O || !target_actor || !target_critic || !O->agent_offset || !O->ids || !O->status || !O->obs || !O->reward)
        return PVE_EINVAL;
#ifdef PVE_HOST_EMULATION
    (void)gamma; (void)stream_;
    return PVE_ESTATE;
#else
    if (target_actor->device != f->device || target_critic->device != f->device) return PVE_EINVAL;
    const int32_t *n_rows_dev = O->agent_offset + f->T.B;
    /* mu'(s'[k]) for the 7 rows of every observation, then Q' (main.py:253-260) */
    int32_t rc = pve_actor_forward_n(target_actor, O->obs, f->out_cap * PVE_OBS_H, n_rows_dev, PVE_OBS_H, f->act7, stream_);
    if (rc != PVE_OK) return rc;
    return nstep_fold(f, O, gamma, target_critic, stream_);
#endif
}

#ifndef PVE_HOST_EMULATION
/* Q' from f->act7, then plan / scan / fold */
static int32_t nstep_fold(pve_nstep *f, const pve_outputs *O, double gamma, pve_critic *target_critic, void *stream_) {
    pve_stream_t stream = (pve_stream_t)stream_;
    const int32_t *n_rows_dev = O->agent_offset + f->T.B;
    const bool fact = f->F.row0 != nullptr;
    int32_t rc = fact ? critic_forward<PVE_OBS_W>(target_critic, O->row0_out, f->act7, f->out_cap, n_rows_dev, f->q, stream)
                      : critic_forward<PVN_OBS>(target_critic, O->obs, f->act7, f->out_cap, n_rows_dev, f->q, stream);
    if (rc != PVE_OK) return rc;
    const unsigned stamp = (unsigned)(++f->pushes);
    const size_t at = (size_t)(stamp % (unsigned)f->T.M) * (size_t)f->out_cap;
    /* this tick's frames belong in slot stamp % M of the frame log: already there if the step wrote them to
     * pve_nstep_obs_slot() / pve_nstep_factored_slot(), copied otherwise (whole blocks: the row count lives on the device) */
    const auto put = [&](void *slot, const void *src, size_t bytes) {
        return slot == src || cudaMemcpyAsync(slot, src, bytes, cudaMemcpyDeviceToDevice, stream) == cudaSuccess;
    };
    const size_t oc = (size_t)f->out_cap;
    const bool ok = fact ? put(f->F.row0 + at * PVE_OBS_W, O->row0_out, oc * PVE_OBS_W * sizeof(float))
                           && put(f->F.prev + at * PVE_OBS_W, O->prev_row0, oc * PVE_OBS_W * sizeof(float))
                           && put(f->F.src + at * 8, O->obs_src, oc * 8 * sizeof(int16_t))
                           && put(f->F.off + (size_t)(stamp % (unsigned)f->T.M) * (f->T.B + 1), O->agent_offset,
                                  (size_t)(f->T.B + 1) * sizeof(int32_t))
                         : put(f->T.log + at * PVN_OBS, O->obs, oc * PVN_OBS * sizeof(float));
    if (!ok) return PVE_ECUDA;
    pvn_plan_kernel<<<f->n_blk, PVN_PLAN_THREADS, 0, stream>>>(f->T, O->ids, O->status, O->agent_offset, f->out_cap, stamp,
                                                              f->plan, f->blk_count, f->counters);
    pvn_scan_kernel<<<1, 1024, 0, stream>>>(f->blk_count, f->blk_base, f->n_blk, f->counters);
    if (f->profiling) cudaEventRecord(f->fold_ev[0], stream);
    if (fact)
        pvn_fold_kernel<true><<<f->fold_blocks, 256, 0, stream>>>(f->T, f->R, O->ids, O->status, O->reward, f->q, O->agent_offset,
                                                                 f->out_cap, stamp, gamma, f->plan, f->blk_base, f->F);
    else
        pvn_fold_kernel<false><<<f->fold_blocks, 256, 0, stream>>>(f->T, f->R, O->ids, O->status, O->reward, f->q, O->agent_offset,
                                                                  f->out_cap, stamp, gamma, f->plan, f->blk_base, f->F);
    if (f->profiling) cudaEventRecord(f->fold_ev[1], stream);
    return cudaGetLastError() == cudaSuccess ? PVE_OK : PVE_ECUDA;
}
#endif

int32_t pve_nstep_push_scene(pve_nstep *f, pve_scene *s, const pve_outputs *O, double gamma, pve_actor *target_actor,
                             pve_critic *target_critic, void *stream_) {
    if (f && f->F.row0) return nstep_refuse(f, "pve_nstep_push_scene: this folder keeps a factored frame log, push with pve_nstep_push_factored");
    if (!f || !s || !O || !target_actor || !target_critic || !O->agent_offset || !O->ids || !O->status || !O->obs
        || !O->reward || !O->nbr_src)
        return PVE_EINVAL;
#ifdef PVE_HOST_EMULATION
    (void)gamma; (void)stream_;
    return PVE_ESTATE;
#else
    if (target_actor->device != f->device || target_critic->device != f->device || s->device != f->device
        || s->cfg.n_envs != f->T.B)
        return PVE_EINVAL;
    pve_stream_t stream = (pve_stream_t)stream_;
    const int B = f->T.B, VCc = s->prm.VC;
    const size_t slots = (size_t)B * VCc;
    if (!f->need || f->scene_slots != slots) {
        cudaFree(f->need); cudaFree(f->mu_prev);
        f->need = nullptr; f->mu_prev = nullptr;
        if (cudaMalloc((void **)&f->need, slots) != cudaSuccess || cudaMalloc((void **)&f->mu_prev, slots * sizeof(float)) != cudaSuccess) {
            cudaGetLastError();
            return PVE_ENOMEM;
        }
        f->scene_slots = slots;
    }
    if (!target_actor->zero_dev) return PVE_ESTATE;      /* computed by pve_actor_create */
    const int32_t *n_rows_dev = O->agent_offset + B;
    const long long rows7 = f->out_cap * PVE_OBS_H;
    if (rows7 > 0x7fffffffLL || (long long)slots > 0x7fffffffLL) return PVE_EINVAL;
    /* 1. this tick's agent rows (row 0 of every observation), written to act7[r][0] in place */
    if (launch_actor(target_actor, O->obs, nullptr, nullptr, nullptr, 0.f, f->act7, PVA_TILE,
                     (int)((f->out_cap + PVA_TILE - 1) / PVA_TILE), f->out_cap, stream, n_rows_dev, 1, nullptr, PVE_OBS_H) != cudaSuccess)
        return PVE_ECUDA;
    /* 2. the rows stored last tick that some observation refers to (the buffer the last step read from) */
    if (cudaMemsetAsync(f->need, 0, slots, stream) != cudaSuccess) return PVE_ECUDA;
    const long long items = f->out_cap * 8;
    const int grid = (int)((items + 255) / 256);
    pvn_mark_kernel<<<grid, 256, 0, stream>>>(O->nbr_src, O->ids, O->agent_offset, B, f->out_cap, VCc, f->need);
    if (launch_actor(target_actor, s->st.row0[s->phase ^ 1], nullptr, nullptr, nullptr, 0.f, f->mu_prev, PVA_TILE,
                     (int)((slots + PVA_TILE - 1) / PVA_TILE), (long long)slots, stream, nullptr, 1, f->need, 1) != cudaSuccess)
        return PVE_ECUDA;
    /* 3. act7[r][1..6] through nbr_src */
    pvn_gather_kernel<<<grid, 256, 0, stream>>>(O->nbr_src, O->ids, O->agent_offset, B, f->out_cap, VCc, f->mu_prev,
                                                target_actor->zero_dev + 28, f->act7);
    if (cudaGetLastError() != cudaSuccess) return PVE_ECUDA;
    return nstep_fold(f, O, gamma, target_critic, stream_);
#endif
}

int32_t pve_nstep_push_factored(pve_nstep *f, const pve_outputs *O, double gamma, pve_actor *target_actor,
                                pve_critic *target_critic, void *stream_) {
    if (f && !f->F.row0) return nstep_refuse(f, "pve_nstep_push_factored: this folder keeps a full-frame log (pve_nstep_create); "
                                                "create it with pve_nstep_create_factored");
    if (f && O && (!O->row0_out || !O->prev_row0 || !O->obs_src))
        return nstep_refuse(f, "pve_nstep_push_factored: the outputs need row0_out, prev_row0 and obs_src");
    if (!f || !O || !target_actor || !target_critic || !O->agent_offset || !O->ids || !O->status || !O->reward)
        return PVE_EINVAL;
#ifdef PVE_HOST_EMULATION
    (void)gamma; (void)stream_;
    return PVE_ESTATE;
#else
    if (target_actor->device != f->device || target_critic->device != f->device) return PVE_EINVAL;
    if (!target_actor->zero_dev) return PVE_ESTATE;      /* computed by pve_actor_create */
    pve_stream_t stream = (pve_stream_t)stream_;
    const int B = f->T.B;
    const int32_t *n_rows_dev = O->agent_offset + B;
    const long long oc = f->out_cap;
    const int groups = (int)((oc + PVA_TILE - 1) / PVA_TILE);
    /* 1. this tick's agent rows (row0_out) */
    if (launch_actor(target_actor, O->row0_out, nullptr, nullptr, nullptr, 0.f, f->mu0, PVA_TILE, groups, oc, stream,
                     n_rows_dev, 1, nullptr, 1) != cudaSuccess)
        return PVE_ECUDA;
    /* 2. the prev_row0 rows that some observation refers to */
    if (cudaMemsetAsync(f->need, 0, (size_t)oc, stream) != cudaSuccess) return PVE_ECUDA;
    const int grid = (int)((oc * 8 + 255) / 256);
    pvn_mark_factored_kernel<<<grid, 256, 0, stream>>>(O->obs_src, O->ids, O->agent_offset, B, oc, f->need);
    if (launch_actor(target_actor, O->prev_row0, nullptr, nullptr, nullptr, 0.f, f->mu_prev, PVA_TILE, groups, oc, stream,
                     n_rows_dev, 1, f->need, 1) != cudaSuccess)
        return PVE_ECUDA;
    /* 3. act7[r][0..6] through obs_src */
    pvn_gather_factored_kernel<<<grid, 256, 0, stream>>>(O->obs_src, O->ids, O->agent_offset, B, oc, f->mu0, f->mu_prev,
                                                         target_actor->zero_dev + 28, f->act7);
    if (cudaGetLastError() != cudaSuccess) return PVE_ECUDA;
    return nstep_fold(f, O, gamma, target_critic, stream_);
#endif
}

int32_t pve_nstep_obs_slot(const pve_nstep *f, float **obs_dev) {
    if (!f || !obs_dev) return PVE_EINVAL;
    *obs_dev = f->T.log ? f->T.log + (size_t)((unsigned)(f->pushes + 1) % (unsigned)f->T.M) * (size_t)f->out_cap * PVN_OBS : nullptr;
    return f->T.log ? PVE_OK : PVE_ESTATE;
}

int32_t pve_nstep_factored_slot(const pve_nstep *f, float **row0_dev, float **prev_dev, int16_t **src_dev) {
    if (!f || !row0_dev || !prev_dev || !src_dev) return PVE_EINVAL;
    if (!f->F.row0) return PVE_ESTATE;
    const size_t at = (size_t)((unsigned)(f->pushes + 1) % (unsigned)f->T.M) * (size_t)f->out_cap;
    *row0_dev = f->F.row0 + at * PVE_OBS_W;
    *prev_dev = f->F.prev + at * PVE_OBS_W;
    *src_dev = f->F.src + at * 8;
    return PVE_OK;
}

int64_t pve_nstep_log_bytes(const pve_nstep *f) {
    if (!f) return PVE_EINVAL;
    const long long M = f->T.M, oc = f->out_cap;
    if (f->F.row0) return M * (oc * (2 * PVE_OBS_W * (long long)sizeof(float) + 8 * (long long)sizeof(int16_t))
                               + (f->T.B + 1) * (long long)sizeof(int32_t));
    return M * oc * PVN_OBS * (long long)sizeof(float);
}

const char *pve_nstep_last_error(const pve_nstep *f) { return f ? f->err : "null folder"; }

int32_t pve_nstep_set_profiling(pve_nstep *f, int32_t on) {
    if (!f) return PVE_EINVAL;
#ifdef PVE_HOST_EMULATION
    (void)on;
    return PVE_ESTATE;
#else
    if (on && !f->profiling) {
        if (cudaEventCreate(&f->fold_ev[0]) != cudaSuccess) return PVE_ECUDA;
        if (cudaEventCreate(&f->fold_ev[1]) != cudaSuccess) { cudaEventDestroy(f->fold_ev[0]); return PVE_ECUDA; }
        f->profiling = 1;
    } else if (!on && f->profiling) {
        cudaEventDestroy(f->fold_ev[0]);
        cudaEventDestroy(f->fold_ev[1]);
        f->profiling = 0;
    }
    return PVE_OK;
#endif
}

int32_t pve_nstep_fold_ms(pve_nstep *f, float *ms) {
    if (!f || !ms) return PVE_EINVAL;
#ifdef PVE_HOST_EMULATION
    return PVE_ESTATE;
#else
    if (!f->profiling || f->pushes == 0) return PVE_ESTATE;
    if (cudaEventSynchronize(f->fold_ev[1]) != cudaSuccess || cudaEventElapsedTime(ms, f->fold_ev[0], f->fold_ev[1]) != cudaSuccess)
        return PVE_ECUDA;
    return PVE_OK;
#endif
}

int32_t pve_nstep_reset(pve_nstep *f, void *stream_) {
    if (!f) return PVE_EINVAL;
#ifdef PVE_HOST_EMULATION
    (void)stream_;
    return PVE_ESTATE;
#else
    const size_t slots = (size_t)f->T.B * f->T.U;
    if (cudaMemsetAsync(f->T.key, 0xFF, slots * 8, (pve_stream_t)stream_) != cudaSuccess
        || cudaMemsetAsync(f->T.fill, 0, slots * 2, (pve_stream_t)stream_) != cudaSuccess)
        return PVE_ECUDA;
    return PVE_OK;
#endif
}

int32_t pve_nstep_replay(const pve_nstep *f, pve_replay_view *view) {
    if (!f || !view) return PVE_EINVAL;
    view->state = f->R.state; view->action = f->R.action; view->reward = f->R.reward;
    view->next_state = f->R.next_state; view->done = f->R.done; view->capacity = f->R.cap;
    return PVE_OK;
}

int32_t pve_nstep_counters(pve_nstep *f, int64_t *out_host, void *stream_) {
    if (!f || !out_host) return PVE_EINVAL;
#ifdef PVE_HOST_EMULATION
    (void)stream_;
    return PVE_ESTATE;
#else
    long long tmp[4];
    if (cudaMemcpyAsync(tmp, f->counters, sizeof(tmp), cudaMemcpyDeviceToHost, (pve_stream_t)stream_) != cudaSuccess
        || cudaStreamSynchronize((pve_stream_t)stream_) != cudaSuccess)
        return PVE_ECUDA;
    out_host[0] = tmp[0]; out_host[1] = tmp[1]; out_host[2] = tmp[2]; out_host[3] = f->pushes;
    return PVE_OK;
#endif
}

const float *pve_nstep_q_dev(const pve_nstep *f) { return f ? f->q : nullptr; }

}  /* extern "C" */
