/*
 * pve_mcc.h -- C ABI of the B200-native batched PVE-MCC environment step.
 *
 * The reference (Mingtzge/PVE-MCC_for_unsignalized_intersection) has no plugin/FFI boundary:
 * its de-facto interface is the Python object `TrafficInteraction` as consumed by main.py.
 * Each entry point below names the reference member it replaces ("TIS" =
 * traffic_interaction_scene.py, "MAIN" = main.py).  One handle = B independent 12-lane
 * intersections resident on one GPU.  All `*_dev` pointers are device pointers (torch
 * `data_ptr()`); `stream` is a `cudaStream_t` passed as `void*`.  No call synchronises the
 * device unless it says so.  Every function returns 0 on success, a negative PVE_E* code
 * otherwise; `pve_last_error()` returns the message.
 *
 * Vehicle slots are DENSE per intersection, ordered (lane ascending, j ascending) -- the order in
 * which MAIN:398-406 iterates `env.veh_info` and therefore the order of the action vector.
 */
#ifndef PVE_MCC_H
#define PVE_MCC_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PVE_NLANE 12
#define PVE_OBS_H 7          /* ego row + 6 neighbour rows        TIS:1295 */
#define PVE_OBS_W 28         /* (6 + 1) * 4 values per row        TIS:1295 */
#define PVE_NNBR 6           /* closer_veh_num / o_agent_num      TIS:187, MAIN:90 */
#define PVE_HDR_BYTES 144    /* packed per-intersection header, see pve_env_header */
#define PVE_NEVER 2147483647 /* spawn tick of an exhausted arrival table */

#define PVE_OK 0
#define PVE_EINVAL -1
#define PVE_ECUDA -2
#define PVE_ENOMEM -3
#define PVE_ESTATE -4

/* status bits of one agent row */
#define PVE_ST_DONE 1        /* veh["Done"] after scene_update            TIS:347, 351 */
#define PVE_ST_REMOVED 2     /* scheduled in delete_veh                   TIS:348      */
#define PVE_ST_FINISHED 4    /* crossed p < 0 this tick; jerk_sum valid   TIS:350-359  */

/* vehicle flag bits inside pve meta.packed (bits 24..31) */
#define PVE_F_CONTROL 1
#define PVE_F_FINISH 2
#define PVE_F_LOCK 4
/* bits 3..4: lock_a + 1 */

/*
 * Construction parameters: replaces TrafficInteraction.__init__ (TIS:21-220, 12-lane branch
 * TIS:146-186).  The geometry constants are supplied by the host so that they are computed
 * with the reference's own expressions (see the Python `SceneConfig`); `pve_default_config`
 * fills them with libm for C callers.
 */
typedef struct pve_config {
    int32_t n_envs;        /* B: intersections on this GPU                                   */
    int32_t veh_cap;       /* dense vehicle slots per intersection (<= 576; rounded up to a class) */
    int32_t agent_cap;     /* controlled vehicles per intersection (<= veh_cap)               */
    int32_t threads;       /* CTA size: 0 = default (128; 512 for the large classes), else 64/96/128/256/512 */
    int64_t out_cap;       /* rows of the per-agent output arrays the caller will provide     */
    double dt, dt2;        /* deltaT and pow(deltaT, 2)                        TIS:21, 1529   */
    double vm, vM, am, aM, v0;                                             /* TIS:21          */
    double collision_thr;  /* args.collision_thr                               TIS:32         */
    double lane_in;        /* lane_info[m][0] = dis_ctl - 6*lane_cw            TIS:149        */
    double lane_len[3];    /* lane_info[m][1]                                  TIS:149-151    */
    double remove_p;       /* -dis_ctl + int((12+1)/2)*lane_cw                 TIS:341-342    */
    double lane_cw;
    /* get_virtual_distance (TIS:733-803) as delta = (p1 - a1) + a2; member iff delta > 0;
     * vd = b + delta.  First index: ego movement 0 = left, 1 = straight; second: k in lane2lane */
    double vd_a1[2][4], vd_a2[2][4], vd_b[2][4];
    double rot_cos[4], rot_sin[4];   /* cos/sin(3.141593/2 * approach)         TIS:1251, 1287 */
    /* != 0: the action of a vehicle whose `control` flag is off is taken as 0 whatever the action array holds --
     * what the reference driver does on the host (`else: action = 0`, MAIN:401-405), for callers that fill every
     * slot without reading the control flags back.  0: actions are used as given (step() semantics, TIS:1502) */
    int32_t zero_uncontrolled;
    /* 0 or 12: the 12-lane intersection (everything above).  4 / 8: the one- / two-lanes-per-approach intersections of
     * the reference's lane_num = 4 and lane_num = 8 branches (TIS:66-99, 100-145) -- SURVEY.md 8(f) row N3: lane_in /
     * lane_len / remove_p above are then those of TIS:53-55 / 101-103 and TIS:341-342, the vd_* and rot_* tables are unused
     * and the n4_* constants below apply.  Lanes 4..11 (8..11) of every [..][12] array (spawn ticks, header) are unused.
     * Vehicles carry their `intention` in bits 5-6 of the flags byte of pve_veh_meta.packed; the 4th value of every
     * observation quad is the ROUTE (direction[lane][intention]).  lane_num = 8 draws every new vehicle's intention at
     * random in the reference (TIS:382, 390); here the draws are an input, see pve_set_intention_draws. */
    int32_t lane_num;
    double n4_T[4][7], n4_C[4][7], n4_C2[4][7];
                                     /* get_virtual_distance (TIS:453-531 / 537-660): member iff p1 - T > 0,
                                      * vd = (|p1 - T| + C) - C2; first index = ego route % 3 (lane_num 4) or % 4 (lane_num 8),
                                      * second = position of the other route in lane2lane */
    double n4_rw[3];                 /* get_state rewrite (TIS:1304-1316, lane_num 4): (alpha' - alpha) 3 cw, alpha' 3 cw, alpha 3 cw */
} pve_config;

/* Per-intersection header as stored on the device (little endian, 144 bytes). */
typedef struct pve_env_header {
    int32_t tick;                 /* scene updates done so far (TIS:223 as an integer)        */
    int32_t id_seq;               /* TIS:212, 433 */
    int32_t passed_veh;           /* TIS:197, 356 */
    int32_t overflow;             /* arrivals dropped because a capacity was reached (sticky) */
    int64_t passed_step_total;    /* TIS:198, 359 */
    int32_t n_veh, n_ctrl;        /* vehicles / controlled vehicles now                       */
    int32_t next_spawn[PVE_NLANE];/* spawn tick of row veh_rec[i] of lane i                   */
    uint16_t veh_rec[PVE_NLANE];  /* TIS:207, 430 */
    uint8_t lane_n[PVE_NLANE];    /* len(veh_info[i]) */
    int8_t head_lane[PVE_NLANE];  /* virtual_lane_4[d][0][1], -1 if the list is empty TIS:1517 */
    uint8_t head_j[PVE_NLANE];    /* virtual_lane_4[d][0][2] (index BEFORE last removal)      */
    uint8_t pad_[4];
} pve_env_header;

/* Per-vehicle integer record: {uid, packed}; packed = step (bits 0..15, saturating) |
 * collision (bits 16..23, saturating) | flags (bits 24..31). */
typedef struct pve_veh_meta { int32_t uid; uint32_t packed; } pve_veh_meta;

/* Raw state for teacher forcing / snapshots (replaces direct access to env.veh_info,
 * SURVEY.md H7).  Pointers may be host or device memory. */
typedef struct pve_state_view {
    pve_env_header *hdr;          /* [B] */
    double *p, *v, *a, *jerk_sum; /* [B][veh_cap]  TIS:403, 410, 411, 405 */
    pve_veh_meta *meta;           /* [B][veh_cap]  */
    float *row0;                  /* [B][veh_cap][28]  veh["state"][0] (TIS:288) */
} pve_state_view;

/*
 * Outputs of one tick: replaces the 9-tuple of scene_update (TIS:376).  Rows of intersection b
 * are agent_offset[b] .. agent_offset[b+1]-1, in the reference's order (lane asc, j asc).
 *   actions  (TIS:290)  == obs[:, :, 2]              estm_collisions (TIS:338) == 0
 *   jerks    (TIS:358)  == jerk_sum[status & FINISHED]
 */
typedef struct pve_outputs {
    int32_t *agent_offset;  /* [B+1]                                                          */
    float *obs;             /* [out_cap][7][28]   re_state                       TIS:289      */
    float *reward;          /* [out_cap]          incl. -10 / +5 overrides       TIS:320-357  */
    int32_t *ids;           /* [out_cap][4]       env, lane, j (pre-removal), uid TIS:291     */
    int32_t *cpv;           /* [out_cap]          collisions_per_veh[k][0]       TIS:339      */
    uint8_t *status;        /* [out_cap]          PVE_ST_* bits                               */
    float *jerk_sum;        /* [out_cap]          veh["jerk_sum"] after the tick TIS:321      */
    int32_t *env_collisions;/* [B]  `collisions`                                 TIS:337      */
    int32_t *env_lock;      /* [B]  `lock`                                       TIS:365-370  */
    int32_t *env_removed;   /* [B]  len(delete_veh)                              TIS:348      */
    /* optional (may be null): [out_cap][8] where each of the 7 observation rows of an agent was copied from
     * (get_state copies whole stored rows, TIS:1330-1334, Q3): -1 = the all-zero row; 0 .. 0x3FFF = row 0 of agent
     * g' of the same intersection THIS tick (output row agent_offset[b] + g'; entry 0 is the agent itself);
     * 0x4000 | k = the row stored LAST tick for vehicle slot k of the same intersection (slot order before this
     * tick's removals; pve_row0_prev_dev until the next step).  Entry 7 is padding (-1).  Lets a consumer evaluate a
     * network once per distinct row.  Every lane_num (12, 8, 4) writes it, with the same codes; a 0x4000 code always
     * names the slot of a vehicle that is an agent of this tick. */
    int16_t *nbr_src;
    /* optional (may be null): [out_cap] pve_agent_record, the per-agent scalars of a row in ONE 16-byte record --
     * what a host-side consumer needs of reward / ids / cpv / status / jerk_sum at 16 instead of 29 bytes per agent
     * (the intersection index is implied by agent_offset).  pve_step_host_async delivers these records. */
    void *packed;
    /* optional (may be null), the FACTORED observation: every observation row is a copy (Q3), so the 7 x 28 block of
     * an agent is determined by two 28-float rows per agent of the same tick and 8 codes.  For output row
     * r = agent_offset[b] + g:
     *   row0_out[r]  = obs[r][0], this tick's row 0 of agent g;
     *   prev_row0[r] = the row 0 stored for agent g's vehicle when the tick started (its actor input; zeros for a
     *                  vehicle that spawned last tick);
     *   obs_src[r][q], q < 7: where obs[r][q] comes from: -1 = the all-zero row; g' (0 .. 0x3FFF) =
     *                  row0_out[agent_offset[b] + g']; 0x4000 | g' = prev_row0[agent_offset[b] + g'].  Entry 0 is g,
     *                  entry 7 is padding (-1).
     * Codes are relative to the agent's own intersection and never refer to another tick's buffers (a neighbour is
     * always an agent of the same tick).  Set all three or none; `obs` may then be null, and the 784 B block of every
     * agent is not written at all.  pve_expand_obs / pve_expand_obs_host rebuild `obs` bit for bit.  lane_num = 12
     * only: with lane_num 4 / 8 pve_step returns PVE_EINVAL when any of them is set. */
    float *row0_out;        /* [out_cap][28] */
    float *prev_row0;       /* [out_cap][28] */
    int16_t *obs_src;       /* [out_cap][8]  */
} pve_outputs;

typedef struct pve_agent_record {
    float reward;           /* as pve_outputs.reward                                           */
    int32_t uid;            /* as ids[3]                                                       */
    uint8_t lane, j;        /* as ids[1], ids[2]                                               */
    uint8_t status;         /* as pve_outputs.status                                           */
    uint8_t cpv;            /* as pve_outputs.cpv, saturating at 255                           */
    float jerk_sum;         /* as pve_outputs.jerk_sum                                         */
} pve_agent_record;

/* End-of-rollout statistics (MAIN:407-415, 566-581), summed over the handle's intersections.
 * Multi-GPU callers all-reduce this 16-double vector (NCCL sum). */
typedef struct pve_counters {
    double agent_steps, vehicle_steps, env_steps, spawned, passed, passed_step_total,
        passed_jerk_sum, collided_agent_steps, lock_events, reward_sum, reward_sq_sum,
        removed, overflow, q5_undefined, reserved0, reserved1;
} pve_counters;

typedef struct pve_scene pve_scene;

const char *pve_backend(void);                 /* "cuda-sm_100a" (or the test-only emulation) */
int32_t pve_default_config(pve_config *cfg, int32_t n_envs, double vm);
int32_t pve_create(const pve_config *cfg, int32_t device, pve_scene **out);
void pve_destroy(pve_scene *s);
const char *pve_last_error(const pve_scene *s);

/* TrafficInteraction(arrive_time, ...) TIS:195-220.  spawn_tick_dev: int32 [B][K][12] built by
 * the host from the arrival tables (SURVEY.md Q8); borrowed, must outlive the rollout.
 * warmup != 0 advances every intersection to its first arrival like TIS:214-220. */
int32_t pve_reset(pve_scene *s, const int32_t *spawn_tick_dev, int32_t K, int32_t warmup, void *stream);

/* A new episode whose traffic the step kernels generate themselves: a Poisson arrival stream per lane, so that no spawn
 * table is built, uploaded or kept (an episode of any length costs O(B) device memory: 192 B per intersection, plus one
 * 32 MB clock table per handle allocated by its first Poisson reset).  For global intersection e = first_env + b, lane i
 * and arrival record r = 0, 1, ...: one Philox4x32-10 block with key (seed & 0xffffffff, seed >> 32) and counter
 * (e, i, r, 0) gives w0..w3; u = (((w0 << 21) | (w1 >> 11)) + 1) * 2^-53; the headway is
 * h_r = max(min_headway, -mean[b][i] * ln(u)) with mean[b][i] = 3600 / rate[b][i] (float64, on the host; here every
 * lane's rate is rate_veh_per_hour, pve_reset_poisson_rates takes one per lane) and ln evaluated by the library's own
 * +-x/ series (bit-identical on every build); T_r = T_{r-1} + h_r in float64 (T_{-1} = 0); the spawn tick is the first
 * n whose accumulated 0.1 s clock (SURVEY.md Q8) is >= T_r, PVE_NEVER past 4 000 000 ticks and from record 65 535 on.
 * lane_num = 8: the intention draw of record r is w2 & 1 (no pve_set_intention_draws needed).  The Python
 * arrivals.poisson_arrivals is the numpy mirror of the stream.
 * Intersections see the same traffic however a batch is sharded: a handle holding intersections [lo, hi) of a larger
 * batch passes first_env = lo. */
typedef struct pve_poisson {
    uint64_t seed;
    double rate_veh_per_hour;   /* finite, > 0 */
    double min_headway;         /* seconds; finite, > 0 (an arrival at 0 s would read as table padding) */
    int64_t first_env;          /* >= 0, first_env + n_envs <= 2^32 */
} pve_poisson;
/* Like pve_reset (state zeroed, warmup != 0 jumps to the first arrival and runs the tick that brings it in), with the
 * arrivals of `p`; nothing is borrowed.  The handle stays in Poisson mode until a pve_reset with a table.  PVE_EINVAL
 * (see pve_last_error) for a rate or min_headway that is not finite and > 0, a negative first_env, first_env + n_envs
 * > 2^32, or pve_config.dt != 0.1. */
int32_t pve_reset_poisson(pve_scene *s, const pve_poisson *p, int32_t warmup, void *stream);
/* pve_reset_poisson with a rate per intersection and lane: rates_host is host memory float64 [n_envs][lane_num] in veh/h,
 * read during the call; p->rate_veh_per_hour is not read.  Everything else of the stream is the same, so rates that are
 * all equal give bit for bit the traffic of pve_reset_poisson at that rate.  A handle holding intersections [lo, hi) of
 * a larger batch passes rates[lo:hi] and first_env = lo.  PVE_EINVAL for a null rates_host, for an entry that is not
 * finite and > 0 (pve_last_error names its intersection and lane), and for the other arguments as pve_reset_poisson.
 * A later pve_reset or pve_reset_poisson replaces the rates. */
int32_t pve_reset_poisson_rates(pve_scene *s, const pve_poisson *p, const double *rates_host, int32_t warmup,
                                void *stream);

/* lane_num = 8 only, before pve_reset: draws_dev uint8 [B][K][12], draws_dev[b][k][i] in {0, 1} = what the reference's
 * `random.randint(0, 1)` returns for the k-th arrival of lane i (TIS:390: intention = self.intention[i][draw]); K and the
 * layout are those of the spawn table handed to the next pve_reset.  Borrowed, must outlive the rollout. */
int32_t pve_set_intention_draws(pve_scene *s, const uint8_t *draws_dev);

/* step(i, j, a) for every vehicle (TIS:1501, MAIN:398-406) + scene_update() (TIS:222) +
 * delete_vehicle() (TIS:435).  actions_dev: float [B][veh_cap]. */
int32_t pve_step(pve_scene *s, const float *actions_dev, const pve_outputs *out_dev, void *stream);

/* Rebuild obs[r] (float [7][28]) from the factored outputs of one tick (pve_outputs.row0_out / prev_row0 / obs_src),
 * bit for bit, for the rows of intersections [b0, b1): rows agent_offset[b0] .. agent_offset[b1] - 1 (agent_offset
 * [b1 + 1] entries).  Like the step, an intersection whose rows do not all fit below `out_cap` is skipped (the step
 * wrote none of its rows).  Plain C on host memory; disjoint intersection ranges may be expanded from different threads
 * at once.  Every code is checked against its own intersection's row count: a row with an invalid code becomes NaN
 * instead of being read out of range.  Returns the number of invalid codes (0 for the output of a step; a negative
 * agent_offset or a decreasing pair of offsets counts as one and skips that intersection), or PVE_EINVAL for a null
 * pointer or b1 < b0. */
int64_t pve_expand_obs_host(const int32_t *agent_offset, int32_t b0, int32_t b1, int64_t out_cap, const float *row0_out,
                            const float *prev_row0, const int16_t *obs_src, float *obs_out);
/* The same for all B intersections on the device: one CUDA kernel on `stream` that reads agent_offset_dev[0 .. B] on
 * the device (nothing waits).  Invalid codes yield NaN rows as above; nothing is counted. */
int32_t pve_expand_obs(const int32_t *agent_offset_dev, int32_t B, int64_t out_cap, const float *row0_out_dev,
                       const float *prev_row0_dev, const int16_t *obs_src_dev, float *obs_dev, void *stream);

/* Same tick through HOST buffers; synchronises.  `copy_mask` bit0: reward/ids/cpv/status/jerk_sum/
 * agent_offset/env_* ; bit1: obs.  `out_host` arrays need `pve_next_agent_total()` rows.
 * Pinned host memory (cudaHostAlloc / cudaHostRegister, torch pin_memory()) is used in place: the kernel reads
 * `actions_host` and writes the bit0 arrays of `out_host` over PCIe while it runs; the bit0 arrays of `out_dev`
 * are then not written this tick (obs always is).  Pageable buffers are staged through device copies. */
int32_t pve_step_host(pve_scene *s, const float *actions_host, const pve_outputs *out_dev,
                      const pve_outputs *out_host, int32_t copy_mask, void *stream);

/* Pipelined host path: the same tick, but nothing waits.  Actions travel by DMA from `actions_host` (pinned), the
 * kernel runs on `stream`, and agent_offset + the per-intersection counters + the 16-byte agent records
 * (out_dev->packed, required) -- with copy_mask bit1 also the observations, with bit2 the factored observation
 * (row0_out, prev_row0, obs_src: 240 B per agent; required in both sets, and out_dev->obs may then be null so that the
 * step does not write the 784 B block at all) -- travel by DMA into `out_host` on an internal copy stream while the
 * caller already enqueues the next ticks.  Three ticks may be in flight: give
 * consecutive calls different `out_dev` / `out_host` buffer sets (three of them, used in turn) and call
 * pve_host_wait() for tick t before the call for tick t + 3.  The call itself only waits for the previous tick's KERNEL
 * (it needs that tick's row count to size the copies). */
int32_t pve_step_host_async(pve_scene *s, const float *actions_host, const pve_outputs *out_dev,
                            const pve_outputs *out_host, int32_t copy_mask, void *stream);
/* waits until the OLDEST tick enqueued by pve_step_host_async has landed in its host buffers; returns its row count
 * (negative: error) */
int64_t pve_host_wait(pve_scene *s);

/* rows the NEXT pve_step will emit (device scan result; synchronises `stream`) */
int64_t pve_next_agent_total(pve_scene *s, void *stream);

/* Teacher forcing: the state of every intersection from `in`.  hdr.next_spawn is not read: it is recomputed from
 * hdr.veh_rec, from the spawn table in table mode and, in Poisson mode, by summing the headways of records
 * 0 .. veh_rec[i] again in record order -- the additions the spawns made, so the pending arrival time and next_spawn are
 * exact and the rollout continues bit for bit. */
int32_t pve_set_state(pve_scene *s, const pve_state_view *in, void *stream);
int32_t pve_get_state(pve_scene *s, const pve_state_view *out, void *stream);

/* device views for a device-side actor: stored row 0 of every slot, and the packed meta */
const float *pve_row0_dev(const pve_scene *s);
/* the other row buffer: after a step, the stored rows that step read (slot order of its start), which the 0x4000 codes of
 * pve_outputs.nbr_src name.  12 lanes: after every step; lane_num 4 / 8: after a step that wrote nbr_src.  Valid until
 * the next step, reset or set_state. */
const float *pve_row0_prev_dev(const pve_scene *s);
const pve_veh_meta *pve_meta_dev(const pve_scene *s);
const pve_env_header *pve_hdr_dev(const pve_scene *s);

int32_t pve_stats(pve_scene *s, pve_counters *out_dev, void *stream);
/* the same statistics PER INTERSECTION, as the step kernel accumulates them on the device: double [B][PVE_ENV_NSTAT] in
 * the order agent_steps, vehicle_steps, collided_agent_steps (MAIN:569-571), lock_events (MAIN:568), passed_jerk_sum
 * (MAIN:567), reward_sum, reward_sq_sum, removed, env_steps, q5_undefined.  Valid after the stream has drained.
 * What they count: vehicle_steps adds the vehicles present when a tick starts, before that tick's arrivals spawn (the
 * vehicles the tick steps); reward_sum / reward_sq_sum add the fp32 rewards of the rows, overrides included, in float64.
 * pve_reset zeroes them, and its warm-up tick (warmup != 0) counts as one env step and nothing else.  pve_set_state
 * leaves them alone: teacher-forced ticks keep adding to the episode's totals.  They describe the simulation, not the
 * emitted rows: the rows of intersections that out_cap left out (overflow) are counted all the same. */
#define PVE_ENV_NSTAT 10
const double *pve_env_stats_dev(const pve_scene *s);

/* measurement aids: CUDA events around the step kernel and the offset scan of the last pve_step
 * (pve_kernel_ms waits for them), launch geometry, struct size for binding checks */
int32_t pve_set_profiling(pve_scene *s, int32_t on);
int32_t pve_kernel_ms(pve_scene *s, float *step_ms, float *scan_ms);
int64_t pve_smem_bytes(const pve_scene *s);
int32_t pve_threads(const pve_scene *s);
/* How a tick is launched.  out[0] = 1: "dual mode" (the default class with the default CTA size): two concurrent
 * kernels per tick -- intersections whose vehicles and due arrivals fit out[1] slots / out[2] agents run in CTAs of
 * out[3] threads with out[4] bytes of shared memory, the few others in CTAs of pve_threads() / pve_smem_bytes() on an
 * internal high-priority stream; results are identical to the single-kernel launch (out[0] = 0; env PVE_DUAL=0). */
int32_t pve_launch_info(const pve_scene *s, int32_t out[8]);
/* capacities actually in use: the requested ones rounded up to a compiled capacity class
 * (128/80, 128/96, 192/128, 384/320, 576/416); every [B][veh_cap] array uses pve_veh_cap() as its stride */
int32_t pve_veh_cap(const pve_scene *s);
int32_t pve_agent_cap(const pve_scene *s);
int32_t pve_config_bytes(void);

/* ---- batched actor inference (SURVEY.md 8(f) N1) ---------------------------------------------
 * Replaces agent.action(state=[veh["state"][0]], sess) of main.py:44/404/563 for every controlled
 * vehicle at once (model_agent_maddpg.py:23-49: LN28 -> Dense64 -> LN -> ReLU -> Dense64 -> LN ->
 * ReLU -> Dense1 -> 3 tanh, fp32).  `weights_host`: PVE_ACTOR_FLOATS floats in this order:
 *   LayerNorm gamma[28], beta[28]; dense kernel[28][64], bias[64]; LayerNorm_1 gamma[64], beta[64];
 *   dense_1 kernel[64][64], bias[64]; LayerNorm_2 gamma[64], beta[64]; dense_2 kernel[64], bias[1].
 *
 * A handle is immutable once created (weights are fixed; a new network is a new handle) and carries the work counters of
 * its kernel: launches of ONE handle must be ordered on one stream (or by events); different handles are independent.
 * Everything derived from the weights (packed fragments, the action of the all-zero row) is complete when
 * pve_actor_create returns. */
#define PVE_ACTOR_FLOATS 6393
typedef struct pve_actor pve_actor;
int32_t pve_actor_create(const float *weights_host, int32_t n_floats, int32_t device, pve_actor **out);
void pve_actor_destroy(pve_actor *a);
/* actions_dev[i] = actor(rows_dev[i][0..27]) for a dense matrix of n_rows observation rows */
int32_t pve_actor_forward(pve_actor *a, const float *rows_dev, int64_t n_rows, float *actions_dev, void *stream);
/* the action tensor of the next pve_step: actions_dev[b][k] = actor(stored row 0 of slot k) for the
 * controlled vehicles of intersection b, 0 elsewhere (main.py:398-404); optional exploration noise
 * `+ noise_scale * noise_dev[b][k]` (main.py:44; noise_dev may be null) */
int32_t pve_act(pve_scene *s, pve_actor *a, const float *noise_dev, float noise_scale, float *actions_dev,
                void *stream);
/* n_ticks x { pve_act; pve_step }: the test drivers' loop main.py:394-441 / 553-575 (policy on every controlled vehicle,
 * step(), scene_update(), delete_vehicle()) enqueued from C, so that a small scene's evaluation is not bound by the
 * caller's per-tick overhead.  `out` receives every tick's outputs in turn (the last tick's remain); the running
 * tallies are those of pve_stats / the per-intersection statistics.  Asynchronous like its two halves. */
int32_t pve_rollout(pve_scene *s, pve_actor *a, int32_t n_ticks, const float *noise_dev, float noise_scale,
                    float *actions_dev, const pve_outputs *out, void *stream);

/* device-side row count: like pve_actor_forward for the first min(max_rows, n_rows_dev[0] * mult) rows of a dense
 * matrix; nothing is read back (used on the 7 rows of every agent's observation: mult = 7, n_rows_dev =
 * &agent_offset[B]) */
int32_t pve_actor_forward_n(pve_actor *a, const float *rows_dev, int64_t max_rows, const int32_t *n_rows_dev,
                            int32_t mult, float *actions_dev, void *stream);

/* ---- n-step return folding + replay writer (SURVEY.md 8(f) N2) --------------------------------
 * Replaces the per-vehicle bookkeeping of the training loop, main.py:243-266, and ReplayBuffer.add with
 * rand_s=True (replay_buffer.py:45-53), for all intersections of a handle at once.
 *
 * Critic = agent_ddpg_target.Q (model_agent_maddpg.py:52-76, 123-125: LN28 -> Dense64 -> LN -> ReLU ->
 * concat(action, 6 other actions) -> Dense64 -> LN -> ReLU -> Dense1, fp32).  `weights_host`: PVE_CRITIC_FLOATS
 * floats in this order: LayerNorm gamma[28], beta[28]; dense kernel[28][64], bias[64]; LayerNorm_1 gamma[64],
 * beta[64]; dense_1 kernel[71][64], bias[64]; LayerNorm_2 gamma[64], beta[64]; dense_2 kernel[64], bias[1]. */
#define PVE_CRITIC_FLOATS 6841
typedef struct pve_critic pve_critic;
int32_t pve_critic_create(const float *weights_host, int32_t n_floats, int32_t device, pve_critic **out);
void pve_critic_destroy(pve_critic *c);
/* q_dev[i] = Q(obs_dev[i][0][0..27], act7_dev[i][0..6]) for i < min(max_rows, n_rows_dev[0]) (n_rows_dev may be
 * null: all max_rows rows).  obs_dev: [max_rows][7][28] observations, only row 0 is read (main.py:257).  (A factored
 * folder's push runs the same network on pve_outputs.row0_out, rows 28 floats apart.) */
int32_t pve_critic_forward(pve_critic *c, const float *obs_dev, const float *act7_dev, int64_t max_rows,
                           const int32_t *n_rows_dev, float *q_dev, void *stream);

/* The replay memory as device arrays: a ring of `capacity` = buffer_size - 1 records (replay_buffer.py:47-53: the
 * reference's deque never holds buffer_size items).  The k-th record ever added (k from 0) sits at k % capacity;
 * the deque, oldest first, is records max(0, N - capacity) .. N - 1 with N = num_experiences. */
typedef struct pve_replay_view {
    float *state;        /* [capacity][7][28]  seq_data[0][0]  main.py:263 */
    float *action;       /* [capacity][7]      seq_data[0][1]              */
    float *reward;       /* [capacity]         r_target        main.py:250-262 */
    float *next_state;   /* [capacity][7][28]  seq_data[0][3]              */
    uint8_t *done;       /* [capacity]         always 0        main.py:264 */
    int64_t capacity;
} pve_replay_view;

typedef struct pve_nstep pve_nstep;
/* n_envs intersections; uid_slots (power of two >= 16, about 2 x the vehicle capacity) history slots per
 * intersection; seq_max_step = args.seq_max_step (main.py:91, <= 14); out_cap = rows of the per-agent output arrays;
 * buffer_size = ReplayBuffer(buffer_size, ...) (main.py:212), buffer_size - 1 >= out_cap */
int32_t pve_nstep_create(int32_t n_envs, int32_t uid_slots, int32_t seq_max_step, int64_t out_cap,
                         int64_t buffer_size, int32_t device, pve_nstep **out);
/* The same folder with a FACTORED frame log: per push slot the factored observation (row0_out f32[out_cap][28],
 * prev_row0 f32[out_cap][28], obs_src i16[out_cap][8], see pve_outputs) and that push's agent_offset[B + 1] -- 240 B per
 * output row instead of the 784 B block (the log is about 0.31 x as large).  Same arguments and checks.  Push it with
 * pve_nstep_push_factored only; the replay memory, counters and bootstrap values are those of a full-frame folder fed
 * the same ticks, bit for bit. */
int32_t pve_nstep_create_factored(int32_t n_envs, int32_t uid_slots, int32_t seq_max_step, int64_t out_cap,
                                  int64_t buffer_size, int32_t device, pve_nstep **out);
void pve_nstep_destroy(pve_nstep *f);
/* main.py:243-266 for the tick whose outputs are in `out_dev` (agent_offset, ids, status, obs, reward are read).
 * The bootstrap term uses the two target networks on this tick's observations.  Asynchronous on `stream`.
 * Full-frame folders only (a factored folder: PVE_EINVAL, see pve_nstep_last_error). */
int32_t pve_nstep_push(pve_nstep *f, const pve_outputs *out_dev, double gamma, pve_actor *target_actor,
                       pve_critic *target_critic, void *stream);
/* The same tick with the scene at hand and out_dev->nbr_src filled in by the step: the target actor is evaluated once
 * per distinct row (this tick's agent rows + the referenced rows stored last tick + the zero row) instead of on all
 * 7 rows of every observation, and the 7 actions are gathered through nbr_src.  The network sees the same row
 * contents, so results are bit-identical to pve_nstep_push when both run the same network kernels (PVE_ACTOR_IMPL /
 * PVE_CRITIC_IMPL set); by default each call picks its kernel by its own row count, and the zero row's action is
 * computed once on one row, so the two may differ within the networks' tolerance.  Every lane_num (12, 8, 4).  Must be called before the scene's next step (last tick's
 * rows are still in place: pve_row0_prev_dev). */
int32_t pve_nstep_push_scene(pve_nstep *f, pve_scene *s, const pve_outputs *out_dev, double gamma,
                             pve_actor *target_actor, pve_critic *target_critic, void *stream);
/* main.py:243-266 for one tick from its FACTORED observation (factored folders only; otherwise, or when one of
 * row0_out / prev_row0 / obs_src is missing, PVE_EINVAL).  Reads agent_offset, ids, status, reward, row0_out, prev_row0
 * and obs_src; out_dev->obs may be null and is never read.  The target actor runs once per distinct row: on row0_out, on
 * the prev_row0 rows some 0x4000 code refers to, and the 7 actions are gathered through obs_src; the target critic runs on
 * row0_out.  Asynchronous; pushes must come in tick order, but since the outputs carry every row the push needs, it
 * does not have to run before the scene's next step (give that step other output buffers). */
int32_t pve_nstep_push_factored(pve_nstep *f, const pve_outputs *out_dev, double gamma, pve_actor *target_actor,
                                pve_critic *target_critic, void *stream);
/* a new episode (main.py:230 builds a new TrafficInteraction every epoch): every vehicle's buffered transitions are
 * dropped, the replay memory and num_experiences are kept (agent1_memory_seq lives across epochs, main.py:212) */
/* Where the NEXT push expects its observations: a block of the folder's frame log ([out_cap][7][28] floats, device).
 * Hand it to the step as pve_outputs.obs and the push finds the frames in place; any other pve_outputs.obs is copied
 * into the log by the push (one out_cap x 784 B device copy).  The log holds the last seq_max_step + 2 pushes: the
 * per-vehicle buffers of main.py:243-246 keep references into it instead of private copies of veh["state"]. */
int32_t pve_nstep_obs_slot(const pve_nstep *f, float **obs_dev);      /* a factored folder: PVE_ESTATE */
/* The factored folder's counterpart: where the NEXT push expects row0_out / prev_row0 / obs_src (device blocks of the
 * log).  Hand them to the step as pve_outputs fields and the push finds them in place; outputs elsewhere are copied in
 * (one device copy of each, sized by out_cap).  The push always copies agent_offset into the slot.  A full-frame folder:
 * PVE_ESTATE. */
int32_t pve_nstep_factored_slot(const pve_nstep *f, float **row0_dev, float **prev_row0_dev, int16_t **obs_src_dev);
/* bytes of the frame log (either format) */
int64_t pve_nstep_log_bytes(const pve_nstep *f);
/* the message of the last refused push */
const char *pve_nstep_last_error(const pve_nstep *f);
/* measurement aids: CUDA events around the fold kernel of every push while on; pve_nstep_fold_ms waits for the last one */
int32_t pve_nstep_set_profiling(pve_nstep *f, int32_t on);
int32_t pve_nstep_fold_ms(pve_nstep *f, float *ms);
int32_t pve_nstep_reset(pve_nstep *f, void *stream);
int32_t pve_nstep_replay(const pve_nstep *f, pve_replay_view *view);
/* out_host[0] = num_experiences (replay_buffer.py:47), [1] = records added by the last push, [2] = history slots
 * claimed while another live vehicle owned them (sticky; must stay 0), [3] = pushes so far.  Synchronises `stream`. */
int32_t pve_nstep_counters(pve_nstep *f, int64_t *out_host, void *stream);
/* device pointer of the bootstrap values Q' of the last push ([out_cap], valid for its agent rows) */
const float *pve_nstep_q_dev(const pve_nstep *f);

#ifdef __cplusplus
}
#endif
#endif
