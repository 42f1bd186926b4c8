/* n-step return folding and replay writer on the device (SURVEY.md section 8(f) N2).
 *
 * Replaces the training driver's per-vehicle bookkeeping after every scene_update, main.py:243-266:
 *
 *     veh["buffer"].append([state_now, actions, reward, state_next, Done])
 *     if Done or veh["count"] > seq_max_step:
 *         r_target = last reward  (+ gamma * Q'(s'[0], mu'(s'[0]), [mu'(s'[1..6])])  unless Done)
 *         for cur in reversed(buffer[:-1]): r_target = cur.reward + gamma * r_target
 *         memory.add(buffer[0].state, buffer[0].actions, r_target, buffer[0].state_next, False)
 *         buffer.pop(0); count -= 1
 *
 * and ReplayBuffer.add with rand_s=True (replay_buffer.py:45-53): a deque that holds at most
 * buffer_size - 1 records.
 *
 * Device layout.  A vehicle is known by (intersection, uid); its history lives in slot uid mod U of its
 * intersection's table (U a power of two, about twice the vehicle capacity):
 *     key    u64   uid << 32 | stamp of the last push that saw it (all ones = free)
 *     fill   u8x2  n = transitions buffered, head = ring index of the oldest state
 *     rew    f32[M]        reward of the transition whose state_next sits at the same ring index
 *     fidx   i32[M]        ring of FRAME REFERENCES, M = seq_max_step + 2: transition i of the buffer is
 *                          (frame[head + i], frame[head + i + 1]) because state_now of a tick is state_next
 *                          of the tick before (TIS:288, main.py:235) or zeros for a new vehicle (TIS:380, reference -1)
 * The frames themselves live once, in a FRAME LOG of the last M pushes' observation blocks ([M][out_cap][7][28]; a
 * reference is a row of the log).  A vehicle is an agent on consecutive ticks, so its M frames were pushed by the last M
 * pushes and the slot that the current push overwrites (push - M) is referenced by nobody.  The step kernel can write a
 * tick's observations straight into the log (pve_nstep_obs_slot: no copy); any other observation buffer is copied in.
 * Round 1 kept a private 14-frame ring per table slot: 11.5 GB per 4 096 intersections and one more 784-byte copy per
 * agent-tick; now the table is 122 bytes per slot (128 MB) and the log 784 B x out_cap x M.
 * A vehicle is an agent on consecutive ticks from its arrival until Done (TIS:419, 336, 353), so "stamp ==
 * previous push" identifies a live history; anything else in the slot is stale and is overwritten.  A slot
 * whose other owner is still live is counted in counters[2] (sticky; size the table with more slots).
 *
 * Three launches per tick after the target networks (actor on all 7 rows of every agent's observation, then
 * pve_critic_kernel):
 *     pvn_plan_kernel  one thread per agent row: table lookup, "emits a record?" flag, block-local prefix
 *     pvn_scan_kernel  one CTA: prefix over the blocks, advances num_experiences
 *     pvn_fold_kernel  one warp per agent row: ring update, return folding in float64, record written at
 *                      its deque position (order of the reference: intersection, lane, j ascending)
 * HBM-bound: per record 2 x 784 B frames in, 2 x 784 + 36 B out = 3.2 KB per agent-tick in steady state (round 1, with
 * the per-slot frame rings: 4.7 KB).
 *
 * FACTORED frame log (pve_nstep_create_factored): the log keeps each push's factored observation instead of its blocks,
 * per slot row0 f32[out_cap][28], prev f32[out_cap][28], src i16[out_cap][8] (pve_outputs.row0_out / prev_row0 /
 * obs_src) and that push's agent_offset[B + 1]: 240 B per row instead of 784.  A frame reference is the same 32-bit
 * log row slot * out_cap + r; its codes are relative to the vehicle's intersection `env`, so the fold resolves code g'
 * as log row slot * out_cap + off_slot[env] + g' and expands the 49 float4 pieces of the frame into the record.
 *
 * The critic (model_agent_maddpg.py:52-76: LN(28) -> Dense 64 -> LN -> ReLU -> concat 7 actions -> Dense 64 ->
 * LN -> ReLU -> Dense 1) reuses the register-tiled fp32 GEMM chain of actor.cuh; fp32 FFMA for the same
 * conditioning reason.  Device only (numpy restatement for tests: oracle/nstep_oracle.py).
 */
#ifndef PVE_NSTEP_CUH
#define PVE_NSTEP_CUH

#include <stdint.h>

#include "pve_mcc.h"
#include "actor.cuh"

/* flat critic parameter layout (floats), see pve_critic_create */
enum { PVC_LN0_G = 0, PVC_LN0_B = 28, PVC_W1 = 56, PVC_B1 = PVC_W1 + 28 * 64, PVC_LN1_G = PVC_B1 + 64,
       PVC_LN1_B = PVC_LN1_G + 64, PVC_W2 = PVC_LN1_B + 64, PVC_B2 = PVC_W2 + 71 * 64, PVC_LN2_G = PVC_B2 + 64,
       PVC_LN2_B = PVC_LN2_G + 64, PVC_W3 = PVC_LN2_B + 64, PVC_B3 = PVC_W3 + 64, PVC_COUNT = PVC_B3 + 1 };
static_assert(PVC_COUNT == PVE_CRITIC_FLOATS, "critic parameter count");
/* the same vector with dense_1/kernel padded to 72 rows (row 71 = 0), as staged in shared memory */
enum { PVC_S_W2 = PVC_W2, PVC_S_B2 = PVC_S_W2 + 72 * 64, PVC_S_LN2_G = PVC_S_B2 + 64, PVC_S_LN2_B = PVC_S_LN2_G + 64,
       PVC_S_W3 = PVC_S_LN2_B + 64, PVC_S_B3 = PVC_S_W3 + 64, PVC_S_COUNT = PVC_S_B3 + 1 };

#define PVN_MAX_M 16                 /* seq_max_step <= 14 */
#define PVN_FREE 0xFFFFFFFFFFFFFFFFull
#define PVN_PLAN_THREADS 256
#define PVN_OBS (PVE_OBS_H * PVE_OBS_W)

struct PvnTable {
    unsigned long long *key;         /* [B][U] */
    uint8_t *fill;                   /* [B][U][2] */
    float *rew;                      /* [B][U][M] */
    int32_t *fidx;                   /* [B][U][M] rows of the frame log, -1 = the all-zero frame */
    float *log;                      /* [M][out_cap][196] observation blocks of the last M pushes */
    long long out_cap;
    int U, M, S, B;
};

struct PvnFactored {                 /* the factored frame log; all null for a full-frame folder (T.log is used) */
    float *row0, *prev;              /* [M][out_cap][28] */
    int16_t *src;                    /* [M][out_cap][8] */
    int32_t *off;                    /* [M][B + 1] agent_offset of the push that wrote the slot */
};

/* the source of one observation row under its factored code (pve_outputs.obs_src) in an intersection of A rows:
 * 0 = the zero row, 1 = row0_out row `idx`, 2 = prev_row0 row `idx` (relative to the intersection), -1 = invalid */
PVE_HD int pve_obs_src_decode(int16_t c, int64_t A, int64_t *idx) {
    if (c == -1) return 0;
    if (c < 0 || (int64_t)(c & 0x3FFF) >= A) return -1;
    *idx = c & 0x3FFF;
    return (c & 0x4000) ? 2 : 1;
}
#define PVE_NAN_BITS 0x7FC00000u      /* an observation row behind an invalid code */

struct PvnReplay {                   /* replay_buffer.py:8-9 as a ring of cap = buffer_size - 1 records */
    float *state, *action, *reward, *next_state;
    uint8_t *done;
    long long cap;
};

#ifdef __CUDACC__
#define PVC_THREADS 128
#define PVC_TILE 128
#define PVC_AS 76                    /* activation row stride: 72 inputs of layer 2, rows 16 apart in different banks */
#define PVC_WPAD ((PVC_S_COUNT + 3) & ~3)
#define PVC_SMEM_BYTES ((PVC_WPAD + PVC_TILE * PVC_AS) * 4)

/* one tile of <= 16 R agents starting at row0: q[row] = Q'(obs[row][0][:], act7[row][:]); STRIDE = floats from one
 * agent's row 0 to the next (PVN_OBS: observation blocks, PVE_OBS_W: pve_outputs.row0_out) */
template <int R, int STRIDE>
__device__ __forceinline__ void pvc_round(const float *__restrict__ w, float *__restrict__ a, const long long row0,
                                          const int n_valid, const float *__restrict__ obs, const float *__restrict__ act7,
                                          float *__restrict__ q) {
    const int tid = threadIdx.x, cg = tid & 7, rg = tid >> 3;
    if (tid < 16 * R) {                                                            /* NET:58-59 */
        float x[28];
        const bool valid = tid < n_valid;
        const long long r = row0 + (valid ? tid : 0);
        const float4 *src = reinterpret_cast<const float4 *>(obs + r * STRIDE);
#pragma unroll
        for (int i = 0; i < 7; ++i) {
            const float4 v = valid ? src[i] : make_float4(0.f, 0.f, 0.f, 0.f);
            x[4 * i] = v.x; x[4 * i + 1] = v.y; x[4 * i + 2] = v.z; x[4 * i + 3] = v.w;
        }
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
        for (int i = 0; i < 28; i += 4) { s0 += x[i]; s1 += x[i + 1]; s2 += x[i + 2]; s3 += x[i + 3]; }
        const float mean = ((s0 + s1) + (s2 + s3)) * (1.f / 28.f);
        s0 = s1 = s2 = s3 = 0.f;
#pragma unroll
        for (int i = 0; i < 28; i += 4) {
            const float d0 = x[i] - mean, d1 = x[i + 1] - mean, d2 = x[i + 2] - mean, d3 = x[i + 3] - mean;
            s0 = fmaf(d0, d0, s0); s1 = fmaf(d1, d1, s1); s2 = fmaf(d2, d2, s2); s3 = fmaf(d3, d3, s3);
        }
        const float rs = rsqrtf(((s0 + s1) + (s2 + s3)) * (1.f / 28.f) + PVA_EPS);
#pragma unroll
        for (int i = 0; i < 28; i += 4) {
            const float4 g = *reinterpret_cast<const float4 *>(w + PVC_LN0_G + i);
            const float4 b = *reinterpret_cast<const float4 *>(w + PVC_LN0_B + i);
            const float i0 = rs * g.x, i1 = rs * g.y, i2 = rs * g.z, i3 = rs * g.w;
            float4 y;
            y.x = fmaf(x[i], i0, fmaf(-mean, i0, b.x)); y.y = fmaf(x[i + 1], i1, fmaf(-mean, i1, b.y));
            y.z = fmaf(x[i + 2], i2, fmaf(-mean, i2, b.z)); y.w = fmaf(x[i + 3], i3, fmaf(-mean, i3, b.w));
            *reinterpret_cast<float4 *>(a + tid * PVC_AS + i) = y;
        }
        float av[8];                                                               /* NET:66: [a, other_a], zero pad */
#pragma unroll
        for (int i = 0; i < 7; ++i) av[i] = valid ? act7[r * 7 + i] : 0.f;
        av[7] = 0.f;
        *reinterpret_cast<float4 *>(a + tid * PVC_AS + 64) = make_float4(av[0], av[1], av[2], av[3]);
        *reinterpret_cast<float4 *>(a + tid * PVC_AS + 68) = make_float4(av[4], av[5], av[6], av[7]);
    }
    __syncthreads();
    float acc[R][8];
    pva_gemm_tile<28, R, PVC_AS>(a, w + PVC_W1, w + PVC_B1, acc, rg, cg);          /* NET:60 */
    pva_tile_ln_relu<R>(acc, w + PVC_LN1_G, w + PVC_LN1_B, cg);                    /* NET:62-64 */
    __syncthreads();
#pragma unroll
    for (int r = 0; r < R; ++r) {
        float *dst = a + (r * 16 + rg) * PVC_AS + cg * 4;
        *reinterpret_cast<float4 *>(dst) = make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]);
        *reinterpret_cast<float4 *>(dst + 32) = make_float4(acc[r][4], acc[r][5], acc[r][6], acc[r][7]);
    }
    __syncthreads();
    pva_gemm_tile<72, R, PVC_AS>(a, w + PVC_S_W2, w + PVC_S_B2, acc, rg, cg);      /* NET:67 */
    pva_tile_ln_relu<R>(acc, w + PVC_S_LN2_G, w + PVC_S_LN2_B, cg);                /* NET:69-71 */
    {   /* Dense 64 -> 1 (NET:73) */
        const float4 u0 = *reinterpret_cast<const float4 *>(w + PVC_S_W3 + cg * 4);
        const float4 u1 = *reinterpret_cast<const float4 *>(w + PVC_S_W3 + 32 + cg * 4);
        float o[R];
#pragma unroll
        for (int r = 0; r < R; ++r)
            o[r] = fmaf(acc[r][0], u0.x, fmaf(acc[r][1], u0.y, fmaf(acc[r][2], u0.z, acc[r][3] * u0.w)))
                   + fmaf(acc[r][4], u1.x, fmaf(acc[r][5], u1.y, fmaf(acc[r][6], u1.z, acc[r][7] * u1.w)));
#pragma unroll
        for (int d = 1; d < 8; d <<= 1)
#pragma unroll
            for (int r = 0; r < R; ++r) o[r] += __shfl_xor_sync(0xffffffffu, o[r], d);
        const int row = cg * 16 + rg;
        float mine = o[0];
#pragma unroll
        for (int r = 1; r < R; ++r) mine = cg == r ? o[r] : mine;
        if (cg < R && row < n_valid) q[row0 + row] = mine + w[PVC_S_B3];
    }
    __syncthreads();
}

/* q[r] for r < min(n_rows_max, n_rows_dev[0]); persistent CTAs stride over tiles of 128 agents */
template <int STRIDE>
__global__ void __launch_bounds__(PVC_THREADS, 3)
pve_critic_kernel(const float *__restrict__ W, const float *__restrict__ obs, const float *__restrict__ act7,
                  float *__restrict__ q, const long long n_rows_max, const int32_t *__restrict__ n_rows_dev) {
    extern __shared__ __align__(16) unsigned char pvc_smem[];
    float *const w = reinterpret_cast<float *>(pvc_smem);
    float *const a = w + PVC_WPAD;
    const int tid = threadIdx.x;
    const long long n_rows = n_rows_dev ? min(n_rows_max, (long long)n_rows_dev[0]) : n_rows_max;
    if ((long long)blockIdx.x * PVC_TILE >= n_rows) return;
    for (int i = tid; i < PVC_S_COUNT; i += PVC_THREADS) {
        float v;
        if (i < PVC_S_W2 + 71 * 64) v = W[i];
        else if (i < PVC_S_B2) v = 0.f;                                            /* the padding row of dense_1 */
        else v = W[i - 64];
        w[i] = v;
    }
    __syncthreads();
    for (long long t0 = (long long)blockIdx.x * PVC_TILE; t0 < n_rows; t0 += (long long)gridDim.x * PVC_TILE) {
        const int n_valid = (int)min((long long)PVC_TILE, n_rows - t0);
        if (n_valid > 64) pvc_round<8, STRIDE>(w, a, t0, n_valid, obs, act7, q);
        else if (n_valid > 32) pvc_round<4, STRIDE>(w, a, t0, n_valid, obs, act7, q);
        else pvc_round<2, STRIDE>(w, a, t0, n_valid, obs, act7, q);
    }
}

/* ---- bootstrap actions once per distinct row (pve_nstep_push_scene) ---------------------------------------------
 * nbr_src (pve_outputs) names the source of every observation row.  mark: which rows stored last tick are referenced at
 * all; gather: act7[r][k] = mu'(source of row k), k = 1..6 (k = 0 was evaluated in place on this tick's agent rows). */
__global__ void __launch_bounds__(256)
pvn_mark_kernel(const int16_t *__restrict__ nbr_src, const int32_t *__restrict__ ids, const int32_t *__restrict__ agent_offset,
                const int B, const long long out_cap, const int VC, uint8_t *__restrict__ need) {
    const long long n_rows = min((long long)agent_offset[B], out_cap);
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long r = i >> 3;
    const int k = (int)(i & 7);
    if (r >= n_rows || k == 0 || k >= PVE_OBS_H) return;
    const int v = nbr_src[r * 8 + k];
    if (v >= 0 && (v & 0x4000)) need[(size_t)ids[r * 4] * VC + (v & 0x3FFF)] = 1;
}
__global__ void __launch_bounds__(256)
pvn_gather_kernel(const int16_t *__restrict__ nbr_src, const int32_t *__restrict__ ids, const int32_t *__restrict__ agent_offset,
                  const int B, const long long out_cap, const int VC, const float *__restrict__ mu_prev,
                  const float *__restrict__ mu_zero, float *__restrict__ act7) {
    const long long n_rows = min((long long)agent_offset[B], out_cap);
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long r = i >> 3;
    const int k = (int)(i & 7);
    if (r >= n_rows || k == 0 || k >= PVE_OBS_H) return;
    const int v = nbr_src[r * 8 + k];
    const int env = ids[r * 4];
    float a;
    if (v < 0) a = mu_zero[0];                                                       /* TIS:1334: the all-zero row */
    else if (v & 0x4000) a = mu_prev[(size_t)env * VC + (v & 0x3FFF)];               /* stored last tick */
    else a = act7[((long long)agent_offset[env] + v) * PVE_OBS_H];                  /* this tick's row 0 of agent v */
    act7[r * PVE_OBS_H + k] = a;
}

/* ---- the same from the factored observation (pve_nstep_push_factored) -------------------------------------------
 * obs_src names every row: mark the prev_row0 rows that some observation refers to; gather act7[r][k], k = 0..6, from
 * mu0 (the actor on row0_out), mu_prev (on the marked prev_row0 rows) and the zero row's action.  A code is checked
 * against its intersection's row count as pve_expand_obs does; an invalid one gathers NaN. */
__device__ __forceinline__ long long pvn_src_row(const int v, const int32_t *__restrict__ agent_offset, const int env,
                                                 const long long out_cap) {
    const long long o0 = agent_offset[env], o1 = min((long long)agent_offset[env + 1], out_cap);
    const long long g = v & 0x3FFF;
    return (o0 >= 0 && o0 + g < o1) ? o0 + g : -1;
}
__global__ void __launch_bounds__(256)
pvn_mark_factored_kernel(const int16_t *__restrict__ obs_src, const int32_t *__restrict__ ids,
                         const int32_t *__restrict__ agent_offset, const int B, const long long out_cap,
                         uint8_t *__restrict__ need) {
    const long long n_rows = min((long long)agent_offset[B], out_cap);
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long r = i >> 3;
    const int k = (int)(i & 7);
    if (r >= n_rows || k == 0 || k >= PVE_OBS_H) return;
    const int v = obs_src[r * 8 + k];
    if (v < 0 || !(v & 0x4000)) return;
    const long long s = pvn_src_row(v, agent_offset, ids[r * 4], out_cap);
    if (s >= 0) need[s] = 1;
}
__global__ void __launch_bounds__(256)
pvn_gather_factored_kernel(const int16_t *__restrict__ obs_src, const int32_t *__restrict__ ids,
                           const int32_t *__restrict__ agent_offset, const int B, const long long out_cap,
                           const float *__restrict__ mu0, const float *__restrict__ mu_prev,
                           const float *__restrict__ mu_zero, float *__restrict__ act7) {
    const long long n_rows = min((long long)agent_offset[B], out_cap);
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long r = i >> 3;
    const int k = (int)(i & 7);
    if (r >= n_rows || k >= PVE_OBS_H) return;
    const int v = obs_src[r * 8 + k];
    float a;
    if (v == -1) a = mu_zero[0];                                                     /* TIS:1334: the all-zero row */
    else {
        const long long s = v < 0 ? -1 : pvn_src_row(v, agent_offset, ids[r * 4], out_cap);
        a = s < 0 ? __int_as_float((int)PVE_NAN_BITS) : (v & 0x4000) ? mu_prev[s] : mu0[s];
    }
    act7[r * PVE_OBS_H + k] = a;
}

/* ---- plan: which rows add a record, and where ------------------------------------------------ */
/* plan[r] = emits | is_new << 1 | (records of earlier rows of the same 256-row block) << 2 */
__global__ void __launch_bounds__(PVN_PLAN_THREADS)
pvn_plan_kernel(const PvnTable T, const int32_t *__restrict__ ids, const uint8_t *__restrict__ status,
                const int32_t *__restrict__ agent_offset, const long long out_cap, const unsigned stamp,
                uint32_t *__restrict__ plan, int32_t *__restrict__ blk_count, long long *__restrict__ counters) {
    __shared__ int warp_sum[PVN_PLAN_THREADS / 32];
    const long long n_rows = min((long long)agent_offset[T.B], out_cap);
    const long long r = (long long)blockIdx.x * PVN_PLAN_THREADS + threadIdx.x;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    bool emit = false, is_new = false;
    if (r < n_rows) {
        const int4 id = reinterpret_cast<const int4 *>(ids)[r];                    /* env, lane, j, uid */
        const unsigned uid = (unsigned)id.w;
        const size_t slot = (size_t)id.x * T.U + (uid & (unsigned)(T.U - 1));
        const unsigned long long k = T.key[slot];
        const unsigned long long live = ((unsigned long long)uid << 32) | (unsigned long long)(stamp - 1u);
        is_new = k != live;
        if (is_new && k != PVN_FREE && (unsigned)(k & 0xFFFFFFFFull) == stamp - 1u)
            atomicAdd(reinterpret_cast<unsigned long long *>(&counters[2]), 1ull);  /* live history of another vehicle */
        const int n_old = is_new ? 0 : T.fill[slot * 2];
        emit = (status[r] & PVE_ST_DONE) != 0 || n_old + 1 > T.S;                   /* main.py:247-248 */
    }
    const unsigned bal = __ballot_sync(0xffffffffu, emit);
    if (lane == 0) warp_sum[wid] = __popc(bal);
    __syncthreads();
    int before = __popc(bal & ((1u << lane) - 1u)), total = 0;
#pragma unroll
    for (int w = 0; w < PVN_PLAN_THREADS / 32; ++w) {
        const int c = warp_sum[w];
        before += w < wid ? c : 0;
        total += c;
    }
    if (r < out_cap) plan[r] = (emit ? 1u : 0u) | (is_new ? 2u : 0u) | ((unsigned)before << 2);
    if (threadIdx.x == 0) blk_count[blockIdx.x] = total;
}

/* blk_base[c] = num_experiences before this tick + records of the blocks before c; counters[0] += total */
__global__ void __launch_bounds__(1024)
pvn_scan_kernel(const int32_t *__restrict__ blk_count, long long *__restrict__ blk_base, const int n_blk,
                long long *__restrict__ counters) {
    __shared__ long long warp_tot[32];
    __shared__ long long carry;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) carry = counters[0];
    __syncthreads();
    for (int c0 = 0; c0 < n_blk; c0 += 1024) {
        const int c = c0 + tid;
        const long long v = c < n_blk ? blk_count[c] : 0;
        long long x = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const long long y = __shfl_up_sync(0xffffffffu, x, d);
            if (lane >= d) x += y;
        }
        if (lane == 31) warp_tot[wid] = x;
        __syncthreads();
        long long pre = carry;
        for (int w = 0; w < wid; ++w) pre += warp_tot[w];
        if (c < n_blk) blk_base[c] = pre + x - v;
        __syncthreads();
        if (tid == 1023) carry = pre + x;
        __syncthreads();
    }
    if (tid == 0) { counters[1] = carry - counters[0]; counters[0] = carry; }
}

/* ---- fold: one warp per agent row ----------------------------------------------------------- */
__device__ __forceinline__ void pvn_copy_frame(float *__restrict__ dst, const float *__restrict__ src, const int lane) {
    const float4 *s4 = reinterpret_cast<const float4 *>(src);
    float4 *d4 = reinterpret_cast<float4 *>(dst);
    const float4 v0 = s4[lane];
    float4 v1 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (lane < 49 - 32) v1 = s4[32 + lane];
    d4[lane] = v0;
    if (lane < 49 - 32) d4[32 + lane] = v1;
}
__device__ __forceinline__ void pvn_zero_frame(float *__restrict__ dst, const int lane) {
    float4 *d4 = reinterpret_cast<float4 *>(dst);
    d4[lane] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (lane < 49 - 32) d4[32 + lane] = make_float4(0.f, 0.f, 0.f, 0.f);
}

/* frame f (a log row, >= 0) of the factored log, expanded into dst as pve_expand_obs does: lane l stores the float4
 * pieces l and l + 32 of the 49.  `env` is the vehicle's intersection; the frame's codes are relative to it in the
 * offsets of the push that wrote the slot.  action != null: also the action column (TIS:290) of the 7 rows. */
__device__ __forceinline__ void pvn_expand_frame(float *__restrict__ dst, const PvnFactored F, const long long out_cap,
                                                 const int B, const long long f, const int env, const int lane,
                                                 float *__restrict__ action) {
    const long long slot = f / out_cap;
    const int32_t *const off = F.off + slot * (B + 1);
    const long long o0 = off[env], o1 = off[env + 1];
    const long long A = (o0 >= 0 && o1 >= o0 && o1 <= out_cap) ? o1 - o0 : 0;   /* rows the step did not write: NaN */
    const int16_t *const src = F.src + f * 8;
    const float4 *const r0 = reinterpret_cast<const float4 *>(F.row0 + (slot * out_cap + o0) * PVE_OBS_W);
    const float4 *const pr = reinterpret_cast<const float4 *>(F.prev + (slot * out_cap + o0) * PVE_OBS_W);
    float4 *const d4 = reinterpret_cast<float4 *>(dst);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int p = lane + 32 * h;
        if (h == 1 && p >= 49) break;
        const int row = p / 7, piece = p - 7 * row;
        int64_t idx = 0;
        const int k = pve_obs_src_decode(src[row], A, &idx);
        float4 v;
        if (k > 0) v = (k == 1 ? r0 : pr)[idx * 7 + piece];
        else { const float w = k == 0 ? 0.f : __int_as_float((int)PVE_NAN_BITS); v = make_float4(w, w, w, w); }
        d4[p] = v;
        if (action && piece == 0) action[row] = v.z;                                /* column 2 of the row */
    }
}

template <bool FACT>
__global__ void __launch_bounds__(256)
pvn_fold_kernel(const PvnTable T, const PvnReplay R, const int32_t *__restrict__ ids, const uint8_t *__restrict__ status,
                const float *__restrict__ reward, const float *__restrict__ q,
                const int32_t *__restrict__ agent_offset, const long long out_cap, const unsigned stamp, const double gamma,
                const uint32_t *__restrict__ plan, const long long *__restrict__ blk_base, const PvnFactored F) {
    const long long n_rows = min((long long)agent_offset[T.B], out_cap);
    const int lane = threadIdx.x & 31;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long r = warp0; r < n_rows; r += n_warps) {
        const int4 id = reinterpret_cast<const int4 *>(ids)[r];
        const unsigned uid = (unsigned)id.w;
        const size_t slot = (size_t)id.x * T.U + (uid & (unsigned)(T.U - 1));
        const uint32_t pl = plan[r];
        const bool emit = pl & 1u, is_new = pl & 2u, done = (status[r] & PVE_ST_DONE) != 0;
        const int M = T.M;
        int n = 0, head = 0;
        if (!is_new) { n = T.fill[slot * 2]; head = T.fill[slot * 2 + 1]; }
        int32_t *const fidx = T.fidx + slot * (size_t)M;
        float *const rew = T.rew + slot * (size_t)M;
        const long long my_row = (long long)(stamp % (unsigned)M) * T.out_cap + r;   /* this tick's observation in the log */
        const float *const obs_r = T.log + my_row * PVN_OBS;
        const float rew_now = reward[r];
        /* append: state_next and reward of this tick (main.py:244-246) */
        int at = head + n + 1; at -= at >= M ? M : 0;
        if (lane == 0) {
            if (is_new) fidx[head] = -1;                                             /* TIS:380 */
            if (!(emit && done)) { fidx[at] = (int32_t)my_row; rew[at] = rew_now; }  /* a Done vehicle never comes back */
        }
        n += 1;
        if (emit) {
            /* rewards of the n buffered transitions, oldest first; the newest is still in a register */
            int ri = head + lane + 1; ri -= ri >= M ? M : 0;
            const float mine = lane < n - 1 ? rew[ri] : rew_now;
            double tgt = (double)rew_now;                                            /* main.py:250-251 */
            if (!done) tgt = tgt + gamma * (double)q[r];                             /* main.py:256-260 */
            for (int i = n - 2; i >= 0; --i)                                         /* main.py:261-262 */
                tgt = (double)__shfl_sync(0xffffffffu, mine, i) + gamma * tgt;
            const long long pos = (blk_base[r / PVN_PLAN_THREADS] + (long long)(pl >> 2)) % R.cap;   /* RB:47-53 */
            int nx = head + 1; nx -= nx >= M ? M : 0;
            /* both references were stored by earlier pushes (n == 1: the next state is this tick's own row) */
            const int f_state = is_new ? -1 : fidx[head];
            if constexpr (FACT) {
                if (f_state < 0) pvn_zero_frame(R.state + pos * PVN_OBS, lane);
                else pvn_expand_frame(R.state + pos * PVN_OBS, F, T.out_cap, T.B, f_state, id.x, lane, nullptr);
                pvn_expand_frame(R.next_state + pos * PVN_OBS, F, T.out_cap, T.B, n == 1 ? my_row : (long long)fidx[nx],
                                 id.x, lane, R.action + pos * PVE_OBS_H);                      /* TIS:290 */
            } else {
                const float *const src_next = n == 1 ? obs_r : T.log + (size_t)fidx[nx] * PVN_OBS;
                if (f_state < 0) pvn_zero_frame(R.state + pos * PVN_OBS, lane);
                else pvn_copy_frame(R.state + pos * PVN_OBS, T.log + (size_t)f_state * PVN_OBS, lane);
                pvn_copy_frame(R.next_state + pos * PVN_OBS, src_next, lane);
                if (lane < PVE_OBS_H) R.action[pos * PVE_OBS_H + lane] = src_next[lane * PVE_OBS_W + 2];   /* TIS:290 */
            }
            if (lane == 0) { R.reward[pos] = (float)tgt; R.done[pos] = 0; }          /* main.py:263-264 */
            head = nx;                                                               /* main.py:265-266 */
            n -= 1;
        }
        if (lane == 0) {
            T.fill[slot * 2] = (uint8_t)n;
            T.fill[slot * 2 + 1] = (uint8_t)head;
            T.key[slot] = done ? PVN_FREE : (((unsigned long long)uid << 32) | (unsigned long long)stamp);
        }
    }
}
#endif  /* __CUDACC__ */
#endif
