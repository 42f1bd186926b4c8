/* The two networks of the policy stage on the fifth-generation tensor cores (tcgen05 + tensor memory, sm_100a):
 * the actor (model_agent_maddpg.py:23-49; contract of actor.cuh) and the critic (model_agent_maddpg.py:52-76; contract
 * of nstep.cuh), both  LN(28) -> Dense 64 -> LN -> ReLU -> Dense 64 -> LN -> ReLU -> Dense 1.
 *
 * Numerics: the bf16 x 3 split of actor_mma.cuh (every fp32 operand = three bf16 numbers, the six products of order
 * <= 2 kept, fp32 accumulation), so the fp32 graph's accuracy is preserved and the parity bound of the tests is the one
 * of the other two implementations.
 *
 * Shape of the work.  One persistent CTA per SM: THREE GROUPS of 128 threads, each group evaluating 128 rows per round
 * with its own operand buffer, its own 64 columns of tensor memory and its own mbarrier, so that one group's tensor-core
 * phases and global-memory latencies hide behind the other groups' epilogues; in the actor four more warps are PRODUCERS
 * (tickets of intersections, meta loads twelve deep, ballot compaction of the controlled slots into a ring in shared
 * memory; ring positions are reserved with an atomic and every entry validates itself) and run ahead of the groups.
 * THREAD r OF A GROUP OWNS ROW r end to end:
 *   - it loads its 28 inputs, applies the first LayerNorm in registers, splits the result and stores the three bf16
 *     operands straight into the K-major, un-swizzled core-matrix layout of a tcgen05 shared-memory descriptor
 *     (core matrix = 8 rows x 16 bytes; a thread's 16 bytes of one K-chunk sit at  chunk * 2048 + r * 16, so a warp's
 *     128-bit stores are contiguous: no bank conflicts, no swizzle needed);
 *   - the group's first warp, converged, issues the split products (an elected lane per instruction) as
 *     tcgen05.mma.cta_group::1.kind::f16  (M = 128, N = 64,
 *     K = 16 per instruction; 12 for the first layer, 27 / 30 for the second) into a 128-lane x 64-column fp32
 *     accumulator in tensor memory and commits them to the group's mbarrier.  The biases ride in the products: input
 *     column 28 (71 in the critic) is the constant 1 and the matching weight row holds the bias; the actor's second
 *     layer, which has no spare column, takes one more K-slice from a constant "ones" block;
 *   - accumulator row r lives in TMEM lane r, which  tcgen05.ld.32x32b  hands to thread r: LayerNorm, ReLU and the
 *     split for the next layer are thread-local -- no shuffles, no shared-memory round trip for the statistics; the
 *     vectors (gamma, beta, last layer) are kernel parameters, i.e. constant-bank operands of the FFMAs.
 * The weights arrive by one bulk copy (cp.async.bulk, 42 KB) that only the first MMA waits for.
 *
 * Shared-memory images (bytes; s = split 0..2 = high, middle, low):
 *   W1[s][chunk 0..3][n 0..63][8 bf16]   = W1[k = 8 chunk + e][n], row 28 = b1                  3 x 4 KB
 *   W2[s][chunk][n][8 bf16]              actor: 8 chunks; critic: 10 chunks, rows 64..70 multiply the 7 actions,
 *                                        row 71 = b2                                              3 x 8 / 10 KB
 *   WB[s][chunk 0..1][n][8 bf16]         actor only: row 0 = b2, the K-slice that meets the ones block    3 x 2 KB
 *   A [group][s][chunk][r 0..127][8 bf16]   the activations of the current layer                 3 x 3 x 16 / 20 KB
 * Descriptors (cute/arch/mma_sm100_desc.hpp): K-major, SWIZZLE_NONE, version 1; stride byte offset = distance of two
 * 8-row groups = 128, leading byte offset = distance of the two 16-byte K-chunks of one K = 16 instruction = 16 x rows
 * (checked on the device both ways: the other reading of the two offsets fails the parity test).
 */
#ifndef PVE_MLP_TC5_CUH
#define PVE_MLP_TC5_CUH

#include "actor_mma.cuh"
#include "nstep.cuh"

/* vectors of one network: a kernel parameter (constant bank) */
struct PvtVecs {
    float ln0_g[28], ln0_b[28], ln1_g[64], ln1_b[64], ln2_g[64], ln2_b[64], w3[64], b3;
};

#define PVT_W1_SPLIT 4096                                  /* bytes of one split of W1: 4 chunks x 64 n x 16 B */
#define PVT_W_BYTES (3 * PVT_W1_SPLIT + 3 * 10240)         /* actor: W1 | W2 3 x 8 KB | WB 3 x 2 KB; critic: W1 | W2 3 x 10 KB */
#define PVT_GROUPS 3
#define PVT_TILE 128
#define PVT_TMEM_COLS 256
#define PVT_RING 4096
#define PVT_MARGIN 1536                                    /* ring slots never handed out: three other producers may reserve at the same time, and the groups free their tiles out of order */
#ifndef PVT_BATCH
#define PVT_BATCH 3                                        /* intersections per ticket */
#endif
#ifndef PVT_PCHUNKS
#define PVT_PCHUNKS 12                                     /* 32-slot chunks a producer loads at once */
#endif
#ifndef PVT_PREFETCH
#define PVT_PREFETCH 1                                     /* draw the next ticket before this one's loads (1) or after its commit (0) */
#endif
#define PVT_PRODUCERS 4                                    /* the register file is handed out four warps at a time: 13 warps cost 16 */
#define PVT_THREADS_ACTOR (PVT_GROUPS * 128 + PVT_PRODUCERS * 32)
#define PVT_THREADS_CRITIC (PVT_GROUPS * 128)

/* host: the shared-memory image of the split weights; W1 = [28][64], W2 = [k2][64] row-major fp32, b1 / b2 = [64] */
static inline void pvt_pack(const float *W1, const float *b1, const float *W2, const float *b2, int critic, uint16_t *out) {
    memset(out, 0, (size_t)PVT_W_BYTES);
    uint16_t *o1 = out, *o2 = out + 3 * PVT_W1_SPLIT / 2;
    const int k2 = critic ? 71 : 64, w2_split = critic ? 5120 : 4096;            /* elements */
    uint16_t *ob = o2 + 3 * w2_split;                                            /* actor: the bias slice */
    for (int n = 0; n < 64; ++n) {
        uint16_t e[3];
        for (int k = 0; k <= 28; ++k) {
            pvm_split3(k < 28 ? W1[k * 64 + n] : b1[n], e);
            for (int s = 0; s < 3; ++s) o1[s * (PVT_W1_SPLIT / 2) + (k / 8) * 512 + n * 8 + (k % 8)] = e[s];
        }
        for (int k = 0; k < k2 + (critic ? 1 : 0); ++k) {
            pvm_split3(k < k2 ? W2[k * 64 + n] : b2[n], e);
            for (int s = 0; s < 3; ++s) o2[s * w2_split + (k / 8) * 512 + n * 8 + (k % 8)] = e[s];
        }
        if (!critic) {
            pvm_split3(b2[n], e);
            for (int s = 0; s < 3; ++s) ob[s * 1024 + n * 8] = e[s];
        }
    }
}
static inline void pvt_vecs_actor(const float *W, PvtVecs *v) {
    memcpy(v->ln0_g, W + PVA_LN0_G, 28 * 4); memcpy(v->ln0_b, W + PVA_LN0_B, 28 * 4);
    memcpy(v->ln1_g, W + PVA_LN1_G, 64 * 4); memcpy(v->ln1_b, W + PVA_LN1_B, 64 * 4);
    memcpy(v->ln2_g, W + PVA_LN2_G, 64 * 4); memcpy(v->ln2_b, W + PVA_LN2_B, 64 * 4);
    memcpy(v->w3, W + PVA_W3, 64 * 4); v->b3 = W[PVA_B3];
}
static inline void pvt_vecs_critic(const float *W, PvtVecs *v) {
    memcpy(v->ln0_g, W + PVC_LN0_G, 28 * 4); memcpy(v->ln0_b, W + PVC_LN0_B, 28 * 4);
    memcpy(v->ln1_g, W + PVC_LN1_G, 64 * 4); memcpy(v->ln1_b, W + PVC_LN1_B, 64 * 4);
    memcpy(v->ln2_g, W + PVC_LN2_G, 64 * 4); memcpy(v->ln2_b, W + PVC_LN2_B, 64 * 4);
    memcpy(v->w3, W + PVC_W3, 64 * 4); v->b3 = W[PVC_B3];
}

#ifdef __CUDACC__

struct PvtCtrl {                       /* in dynamic shared memory, after the buffers */
    uint64_t wbar;                     /* the weights have landed */
    uint64_t mbar[PVT_GROUPS];         /* a group's products are complete */
    uint32_t tmem_slot;
    int q_res, q_head, q_free, q_done; /* ring positions reserved by the producers / claimed by the groups / read and cleared; all producers done */
    int p_done;                        /* producers that have finished */
    int grp_head[PVT_GROUPS], grp_n[PVT_GROUPS];
};
#define PVT_A_SPLIT(CRITIC) ((CRITIC) ? 20480 : 16384)
#define PVT_ONES_BYTES 4096
#define PVT_ACTOR_SMEM (PVT_W_BYTES + PVT_ONES_BYTES + PVT_GROUPS * 3 * PVT_A_SPLIT(0) + PVT_RING * 4 + (int)sizeof(PvtCtrl))
#define PVT_CRITIC_SMEM (PVT_W_BYTES + PVT_GROUPS * 3 * PVT_A_SPLIT(1) + (int)sizeof(PvtCtrl))

/* ---- PTX wrappers ---------------------------------------------------------------------------------- */
__device__ __forceinline__ uint32_t pvt_saddr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

/* K-major, no swizzle, sm_100 descriptor version 1: leading byte offset = K-chunk distance, stride byte offset = 128 */
__device__ __forceinline__ uint64_t pvt_desc(uint32_t saddr, uint32_t kchunk) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)((kchunk >> 4) & 0x3FFFu) << 16)
           | ((uint64_t)(128u >> 4) << 32) | (1ull << 46);
}
/* D (fp32, TMEM) (+)= A (bf16, smem) x B (bf16, smem); M = 128, N = 64 */
#define PVT_IDESC ((1u << 4) | (1u << 7) | (1u << 10) | ((64u >> 3) << 17) | ((128u >> 4) << 24))
/* The issuing warp runs converged with warp-uniform operands and elects one lane per instruction (the same lane every
 * time), so that the descriptors live in uniform registers: issued from a single diverged thread, every tcgen05.mma
 * cost ~16 instructions and ~100 cycles (a broadcast loop over the active lanes), 2 us of a 7.5 us round. */
__device__ __forceinline__ bool pvt_elect() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}\n" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void pvt_mma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t accumulate) {
#ifdef PVT_X_NOMMA                      /* experiment: the kernel without its tensor-core work (results are garbage) */
    return;
#endif
    if (pvt_elect())
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                     "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
                     :: "r"(tmem_d), "l"(da), "l"(db), "r"(PVT_IDESC), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void pvt_commit(uint32_t bar) {
    if (pvt_elect())
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar) : "memory");
}
__device__ __forceinline__ void pvt_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void pvt_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void pvt_fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void pvt_gsync(int id) { asm volatile("bar.sync %0, 128;" :: "r"(id) : "memory"); }
/* a hang here would cost a GPU box: anything that does not complete within ~2 s traps instead */
#define PVT_TIMEOUT(t0) do { if (clock64() - (t0) > 4000000000LL) __trap(); } while (0)
__device__ __forceinline__ void pvt_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    for (int spins = 0;; ++spins) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if (done) break;
        if (spins > (1 << 24)) __trap();
    }
}
#define PVT_LD16(r, o, taddr)                                                                                          \
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];" \
                 : "=r"(r[o + 0]), "=r"(r[o + 1]), "=r"(r[o + 2]), "=r"(r[o + 3]), "=r"(r[o + 4]), "=r"(r[o + 5]),       \
                   "=r"(r[o + 6]), "=r"(r[o + 7]), "=r"(r[o + 8]), "=r"(r[o + 9]), "=r"(r[o + 10]), "=r"(r[o + 11]),     \
                   "=r"(r[o + 12]), "=r"(r[o + 13]), "=r"(r[o + 14]), "=r"(r[o + 15])                                    \
                 : "r"((taddr) + (o)))
/* the 64 accumulator columns of this thread's row; taddr = group's columns | (32 (warp % 4)) << 16 */
__device__ __forceinline__ void pvt_load_row(float (&v)[64], uint32_t taddr) {
    uint32_t r[64];
    PVT_LD16(r, 0, taddr); PVT_LD16(r, 16, taddr); PVT_LD16(r, 32, taddr); PVT_LD16(r, 48, taddr);
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int j = 0; j < 64; ++j) v[j] = __uint_as_float(r[j]);
}

/* (x0, x1) -> three bf16x2 words, x0 in the low half (the lower k index); x = high + middle + low up to 2^-24 */
__device__ __forceinline__ void pvt_split_pair(float x0, float x1, uint32_t &h, uint32_t &m, uint32_t &l) {
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(h) : "f"(x1), "f"(x0));
    const float r0 = x0 - __uint_as_float(h << 16), r1 = x1 - __uint_as_float(h & 0xffff0000u);
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(m) : "f"(r1), "f"(r0));
    const float q0 = r0 - __uint_as_float(m << 16), q1 = r1 - __uint_as_float(m & 0xffff0000u);
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(l) : "f"(q1), "f"(q0));
}
/* eight consecutive values of this thread's row -> one 16-byte K-chunk of each of the three operands */
__device__ __forceinline__ void pvt_store_chunk(unsigned char *a, int a_split, int chunk, int row, const float *y) {
    uint4 h, m, l;
    pvt_split_pair(y[0], y[1], h.x, m.x, l.x); pvt_split_pair(y[2], y[3], h.y, m.y, l.y);
    pvt_split_pair(y[4], y[5], h.z, m.z, l.z); pvt_split_pair(y[6], y[7], h.w, m.w, l.w);
    unsigned char *p = a + chunk * 2048 + row * 16;
    *reinterpret_cast<uint4 *>(p) = h;
    *reinterpret_cast<uint4 *>(p + a_split) = m;
    *reinterpret_cast<uint4 *>(p + 2 * a_split) = l;
}

#ifndef PVT_X_PRODUCTS
#define PVT_X_PRODUCTS 6               /* experiment knob: fewer products (results lose accuracy) */
#endif
/* one thread: the six split products over KSTEPS K = 16 slices, small terms first (as pvm_kstep);
 * a / b = descriptors of split 0, chunk 0 */
template <int KSTEPS>
__device__ __forceinline__ void pvt_issue(uint32_t tmem, uint64_t a, uint32_t a_split, uint64_t b, uint32_t b_split, bool fresh) {
#pragma unroll
    for (int p = 0; p < PVT_X_PRODUCTS; ++p) {
        const int sa = p == 0 ? 2 : (p == 1 || p == 3) ? 1 : 0;      /* al bh, am bm, ah bl, am bh, ah bm, ah bh */
        const int sb = (p == 0 || p == 3 || p == 5) ? 0 : (p == 1 || p == 4) ? 1 : 2;
#pragma unroll
        for (int kk = 0; kk < KSTEPS; ++kk)
            pvt_mma(tmem, a + ((sa * a_split + kk * 4096) >> 4), b + ((sb * b_split + kk * 2048) >> 4),      /* start-address field */
                    (!fresh || (p | kk) != 0) ? 1u : 0u);
    }
}

/* LayerNorm + ReLU of this thread's row (the bias is already in v): mean, centred second moment, then
 * (v - mean) (rsqrt gamma) + beta -- algebraically the reference's x inv + (beta - mean inv) */
__device__ __forceinline__ void pvt_ln_relu(float (&v)[64], const float *gamma, const float *beta) {
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
    for (int j = 0; j < 64; j += 4) { s0 += v[j]; s1 += v[j + 1]; s2 += v[j + 2]; s3 += v[j + 3]; }
    const float mean = ((s0 + s1) + (s2 + s3)) * (1.f / 64.f);
    float q0 = 0.f, q1 = 0.f, q2 = 0.f, q3 = 0.f;
#pragma unroll
    for (int j = 0; j < 64; j += 4) {
        v[j] -= mean; v[j + 1] -= mean; v[j + 2] -= mean; v[j + 3] -= mean;
        q0 = fmaf(v[j], v[j], q0); q1 = fmaf(v[j + 1], v[j + 1], q1); q2 = fmaf(v[j + 2], v[j + 2], q2); q3 = fmaf(v[j + 3], v[j + 3], q3);
    }
    const float rs = rsqrtf(((q0 + q1) + (q2 + q3)) * (1.f / 64.f) + PVA_EPS);
#pragma unroll
    for (int j = 0; j < 64; ++j) v[j] = fmaxf(fmaf(v[j], rs * gamma[j], beta[j]), 0.f);
}

#ifdef PVT_X_TRACE                     /* experiment: clock64 stamps of the first rounds of the first CTAs (tools/actor_trace.py) */
__device__ long long pvt_trace_buf[8 * 3 * 16 * 12];
#define PVT_STAMP(G, ev) do { if ((G).tr && (G).gt == 0) (G).tr[ev] = clock64(); } while (0)
#else
#define PVT_STAMP(G, ev) do { } while (0)
#endif
/* what a group needs for its rounds */
struct PvtGroup {
    unsigned char *a;                  /* the group's operand buffer: [3 splits][chunks][128 rows][16 B] */
    uint64_t da, dw1, dw2, dwb, dones; /* descriptors (split 0, chunk 0): operand buffer, W1, W2, bias slice, ones block */
    uint32_t taddr;                    /* tensor memory: the group's 64 columns, this warp's 32 lanes */
    uint32_t bar, wbar, parity;
    int id, gt;                        /* named barrier of the group, thread in group */
    bool w_ready, lead;                /* lead: this warp issues the group's products (warp-uniform by construction) */
    long long *tr;                     /* PVT_X_TRACE: this round's stamps */
};

/* One round: row `src` (28 floats, or nullptr for a padding row) of every thread of the group through the network.
 * Returns the last layer's h2 . w3 + b3.  The 128 threads of the group call it together. */
template <bool CRITIC>
__device__ __forceinline__ float pvt_round(const PvtVecs &V, PvtGroup &G, const float *__restrict__ src, const float *__restrict__ act) {
    constexpr int A_SPLIT = PVT_A_SPLIT(CRITIC), W2_SPLIT = CRITIC ? 10240 : 8192;
    /* first LayerNorm (NET:27 / NET:58-59); input column 28 = 1 carries the first bias */
    {
        float x[32];
#pragma unroll
        for (int q = 0; q < 7; ++q) {
            const float4 t = src ? reinterpret_cast<const float4 *>(src)[q] : make_float4(0.f, 0.f, 0.f, 0.f);
            x[4 * q] = t.x; x[4 * q + 1] = t.y; x[4 * q + 2] = t.z; x[4 * q + 3] = t.w;
        }
        float s = 0.f;
#pragma unroll
        for (int q = 0; q < 7; ++q) s += (x[4 * q] + x[4 * q + 1]) + (x[4 * q + 2] + x[4 * q + 3]);
        const float mean = s * (1.f / 28.f);
        float q2 = 0.f;
#pragma unroll
        for (int k = 0; k < 28; ++k) { x[k] -= mean; q2 = fmaf(x[k], x[k], q2); }
        const float rs = rsqrtf(q2 * (1.f / 28.f) + PVA_EPS);
#pragma unroll
        for (int k = 0; k < 28; ++k) x[k] = fmaf(x[k], rs * V.ln0_g[k], V.ln0_b[k]);
        x[28] = 1.f; x[29] = x[30] = x[31] = 0.f;
#pragma unroll
        for (int c = 0; c < 4; ++c) pvt_store_chunk(G.a, A_SPLIT, c, G.gt, x + 8 * c);
        if (CRITIC) {                  /* inputs 64..70 of the second layer: the seven actions (NET:66); 71: the bias */
            float y[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) y[i] = i < 7 ? (act ? act[i] : 0.f) : (i == 7 ? 1.f : 0.f);
            pvt_store_chunk(G.a, A_SPLIT, 8, G.gt, y);
            pvt_store_chunk(G.a, A_SPLIT, 9, G.gt, y + 8);
        }
    }
    PVT_STAMP(G, 2);
    pvt_fence_async_smem();            /* generic-proxy stores -> visible to the tensor core's async proxy */
    pvt_fence_before();                /* last round's tcgen05.ld of these TMEM columns is ordered before the barrier */
    pvt_gsync(G.id);
    const uint32_t tmem = G.taddr & 0x0000FFFFu;                       /* lane 0 of the group's columns */
    if (G.lead) {                      /* the group's first warp, converged */
        pvt_fence_after();
        if (!G.w_ready) { pvt_wait(G.wbar, 0); G.w_ready = true; }
        PVT_STAMP(G, 3);
        pvt_issue<2>(tmem, G.da, A_SPLIT, G.dw1, PVT_W1_SPLIT, true);
        pvt_commit(G.bar);
        PVT_STAMP(G, 4);
    }
    pvt_wait(G.bar, G.parity); G.parity ^= 1u;
    PVT_STAMP(G, 5);
    __syncwarp();
    pvt_fence_after();
    float v[64];
    pvt_load_row(v, G.taddr);
    PVT_STAMP(G, 6);
    pvt_ln_relu(v, V.ln1_g, V.ln1_b);                          /* NET:28-32 / 60-64 */
#pragma unroll
    for (int c = 0; c < 8; ++c) pvt_store_chunk(G.a, A_SPLIT, c, G.gt, v + 8 * c);
    PVT_STAMP(G, 7);
    pvt_fence_async_smem();
    pvt_fence_before();
    pvt_gsync(G.id);
    if (G.lead) {
        pvt_fence_after();
        PVT_STAMP(G, 8);
        if (CRITIC) {
            pvt_issue<5>(tmem, G.da, A_SPLIT, G.dw2, W2_SPLIT, true);
        } else {                       /* the second bias: ones block x (low, middle, high) of the bias slice */
            pvt_mma(tmem, G.dones, G.dwb + ((2 * 2048) >> 4), 0u);
            pvt_mma(tmem, G.dones, G.dwb + (2048 >> 4), 1u);
            pvt_issue<4>(tmem, G.da, A_SPLIT, G.dw2, W2_SPLIT, false);
            pvt_mma(tmem, G.dones, G.dwb, 1u);
        }
        pvt_commit(G.bar);
    }
    pvt_wait(G.bar, G.parity); G.parity ^= 1u;
    PVT_STAMP(G, 9);
    __syncwarp();
    pvt_fence_after();
    pvt_load_row(v, G.taddr);
    pvt_ln_relu(v, V.ln2_g, V.ln2_b);                          /* NET:34-38 / 67-71 */
    float o0 = 0.f, o1 = 0.f, o2 = 0.f, o3 = 0.f;              /* Dense 64 -> 1 (NET:40 / 73) */
#pragma unroll
    for (int j = 0; j < 64; j += 4) {
        o0 = fmaf(v[j], V.w3[j], o0); o1 = fmaf(v[j + 1], V.w3[j + 1], o1);
        o2 = fmaf(v[j + 2], V.w3[j + 2], o2); o3 = fmaf(v[j + 3], V.w3[j + 3], o3);
    }
    return ((o0 + o1) + (o2 + o3)) + V.b3;
}

/* prologue shared by the two kernels: barriers, bulk copy of the weight image, tensor-memory allocation.
 * Ends with a CTA-wide barrier; G is filled for threads of the groups (warp < 4 PVT_GROUPS). */
template <bool CRITIC>
__device__ __forceinline__ void pvt_setup(unsigned char *smem, const uint16_t *__restrict__ PW, PvtCtrl *C, PvtGroup &G, uint32_t &tmem) {
    const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);           /* provably warp-uniform */
    unsigned char *const abuf = smem + PVT_W_BYTES + (CRITIC ? 0 : PVT_ONES_BYTES);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(pvt_saddr(&C->wbar)) : "memory");
        for (int g = 0; g < PVT_GROUPS; ++g)
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(pvt_saddr(&C->mbar[g])) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        pvt_fence_async_smem();
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(pvt_saddr(&C->wbar)), "r"((uint32_t)PVT_W_BYTES) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     :: "r"(pvt_saddr(smem)), "l"(PW), "r"((uint32_t)PVT_W_BYTES), "r"(pvt_saddr(&C->wbar)) : "memory");
        C->q_res = 0; C->q_head = 0; C->q_free = 0; C->q_done = 0; C->p_done = 0;
    }
    if (!CRITIC)                       /* ones block: [2 chunks][128 rows][8 bf16], element (row, 0) = 1 */
        for (int i = tid; i < PVT_ONES_BYTES / 16; i += blockDim.x)
            reinterpret_cast<uint4 *>(smem + PVT_W_BYTES)[i] = make_uint4(i < 128 ? 0x3F80u : 0u, 0u, 0u, 0u);
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(pvt_saddr(&C->tmem_slot)), "r"(PVT_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    pvt_fence_async_smem();
    pvt_fence_before();
    __syncthreads();
    pvt_fence_after();
    tmem = *reinterpret_cast<volatile uint32_t *>(&C->tmem_slot);
    const int g = warp >> 2;
    if (g < PVT_GROUPS) {
        G.a = abuf + g * 3 * PVT_A_SPLIT(CRITIC);
        const uint32_t w = pvt_saddr(smem), w2 = w + 3 * PVT_W1_SPLIT;
        G.da = pvt_desc(pvt_saddr(G.a), 2048); G.dw1 = pvt_desc(w, 1024); G.dw2 = pvt_desc(w2, 1024);
        G.dwb = pvt_desc(w2 + 3 * 8192, 1024); G.dones = pvt_desc(w + PVT_W_BYTES, 2048);
        G.taddr = tmem + 64u * g + ((uint32_t)((warp & 3) * 32) << 16);
        G.bar = pvt_saddr(&C->mbar[g]); G.wbar = pvt_saddr(&C->wbar); G.parity = 0;
        G.id = 1 + g; G.gt = tid & 127; G.w_ready = false; G.lead = (warp & 3) == 0; G.tr = nullptr;
    }
}
__device__ __forceinline__ void pvt_teardown(uint32_t tmem) {
    pvt_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) {
        pvt_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(PVT_TMEM_COLS) : "memory");
    }
}

/* ---- actor: same contract as pve_actor_kernel (actor.cuh); PW = pvt_pack's image ------------------------ */
__global__ void __launch_bounds__(PVT_THREADS_ACTOR, 1)
pve_actor_tc_kernel(const __grid_constant__ PvtVecs V, const uint16_t *__restrict__ PW, const float *__restrict__ rows,
                    const pve_veh_meta *__restrict__ meta, const int32_t *__restrict__ n_veh, const float *__restrict__ noise,
                    const float noise_scale, float *__restrict__ actions, const int slots_per_env, const int n_env,
                    const long long n_slots_max, int *__restrict__ ticket, const int32_t *__restrict__ limit_dev,
                    const int limit_mult, const uint8_t *__restrict__ mask, const int slot_step) {
    const long long n_slots = limit_dev ? min(n_slots_max, (long long)limit_dev[0] * limit_mult) : n_slots_max;
    extern __shared__ __align__(128) unsigned char pvt_smem[];
    int *const ring = reinterpret_cast<int *>(pvt_smem + PVT_W_BYTES + PVT_ONES_BYTES + PVT_GROUPS * 3 * PVT_A_SPLIT(0));
    PvtCtrl *const C = reinterpret_cast<PvtCtrl *>(ring + PVT_RING);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t tmem;
    PvtGroup G;
    for (int i = tid; i < PVT_RING; i += PVT_THREADS_ACTOR) ring[i] = -1;       /* empty; ordered by the barrier inside pvt_setup */
    pvt_setup<false>(pvt_smem, PW, C, G, tmem);

    if (warp < 4 * PVT_GROUPS) {
        /* ---- a group: claim up to 128 queued slots, evaluate, store ---- */
        const int g = warp >> 2;
        for (int round = 0;; ++round) {
#ifdef PVT_X_TRACE
            G.tr = (blockIdx.x < 8 && round < 16) ? pvt_trace_buf + ((blockIdx.x * 3 + g) * 16 + round) * 12 : nullptr;
#endif
            PVT_STAMP(G, 0);
            if (G.gt == 0) {
                int h, n;
                const long long t0 = clock64();
                for (;;) {
                    const int done = *reinterpret_cast<volatile int *>(&C->q_done);      /* before the count: a set flag means it is final */
                    __threadfence_block();
                    const int t = *reinterpret_cast<volatile int *>(&C->q_res);
                    h = *reinterpret_cast<volatile int *>(&C->q_head);
                    const int avail = t - h;
                    n = avail >= PVT_TILE ? PVT_TILE : (done ? avail : -1);
                    if (n == 0) break;
                    if (n > 0) { if (atomicCAS(&C->q_head, h, h + n) == h) break; continue; }
                    __nanosleep(200);
                    PVT_TIMEOUT(t0);
                }
                __threadfence_block();
                C->grp_head[g] = h; C->grp_n[g] = n;
            }
            pvt_gsync(G.id);
            const int n_valid = *reinterpret_cast<volatile int *>(&C->grp_n[g]), head = *reinterpret_cast<volatile int *>(&C->grp_head[g]);
            if (n_valid == 0) break;
            const bool valid = G.gt < n_valid;
            long long gs = 0;
            if (valid) {                                             /* the position is reserved; its entry may still be on its way */
                volatile int *const e = ring + ((head + G.gt) & (PVT_RING - 1));
                int v = *e;
                if (v < 0) {
                    const long long t0 = clock64();
                    while ((v = *e) < 0) { __nanosleep(20); PVT_TIMEOUT(t0); }
                }
                *e = -1;
                gs = v;
            }
            pvt_gsync(G.id);                                         /* the ring entries and the claim have been read */
            if (G.gt == 0) atomicAdd(&C->q_free, n_valid);
            PVT_STAMP(G, 1);
            const float o = pvt_round<false>(V, G, valid ? rows + gs * PVE_OBS_W : nullptr, nullptr);
            if (valid) {
                float act = 3.f * tanhf(o);                                  /* NET:40-47 */
                if (noise) act += noise_scale * noise[gs];                   /* main.py:44 */
                actions[gs] = act;
            }
            PVT_STAMP(G, 10);
        }
    } else {
        /* ---- a producer warp: controlled slots of PVT_BATCH intersections per ticket -> ring.  The four producers work
         * independently: a producer reserves ring positions with one atomic and fills them; an entry validates itself (>= 0),
         * so nobody waits for a turn (appending in ticket order cost ~0.6 us per producer at the start, one after the other,
         * while two of the three groups had nothing to claim). ---- */
        const int cpe = (slots_per_env + 31) >> 5;                               /* 32-slot chunks per intersection */
        const unsigned lt = (1u << lane) - 1u;
        /* the first ticket of every producer is static (no round trip to the ticket counter before the first loads),
         * the others are drawn from ticket[0] and start behind the static ones */
        const int pw = warp - 4 * PVT_GROUPS, dyn0 = (int)gridDim.x * PVT_PRODUCERS * PVT_BATCH;
        int tk = ((int)blockIdx.x * PVT_PRODUCERS + pw) * PVT_BATCH;
        bool first = true;
        while (first || tk < n_env) {
            const int envb = tk;
            int ntk = 0;
            if (PVT_PREFETCH && lane == 0) ntk = dyn0 + atomicAdd(&ticket[0], PVT_BATCH);    /* the next ticket travels meanwhile */
            const int n_e = max(0, min(n_env, envb + PVT_BATCH) - envb);
            const int nvl = (meta && lane < n_e) ? n_veh[envb + lane] : slots_per_env;
            const int n_chunks = n_e * cpe;
            int e = 0, c = 0;
            for (int q0 = 0; q0 < n_chunks; q0 += PVT_PCHUNKS) {
                uint32_t pk[PVT_PCHUNKS]; bool pre[PVT_PCHUNKS]; int gi[PVT_PCHUNKS], sv[PVT_PCHUNKS], nvu[PVT_PCHUNKS];
#pragma unroll
                for (int u = 0; u < PVT_PCHUNKS; ++u) {                          /* all loads in flight together */
                    const int s = 32 * c + lane;
                    const long long gs = (long long)(envb + e) * slots_per_env + s;
                    pre[u] = q0 + u < n_chunks && s < slots_per_env && gs < n_slots;
                    if (pre[u] && mask) pre[u] = mask[gs] != 0;                  /* only the marked rows */
                    pk[u] = (pre[u] && meta) ? meta[gs].packed : 0u;
                    gi[u] = (int)gs; sv[u] = s; nvu[u] = e;                     /* the intersection; its vehicle count after the loads */
                    if (++c == cpe) { c = 0; ++e; }
                }
                unsigned bal[PVT_PCHUNKS]; int cnt = 0;
#pragma unroll
                for (int u = 0; u < PVT_PCHUNKS; ++u) {
                    bool want = pre[u];
                    nvu[u] = __shfl_sync(0xffffffffu, nvl, nvu[u] & 31);
                    if (meta) {
                        want = pre[u] && sv[u] < nvu[u] && ((pk[u] >> 24) & PVE_F_CONTROL) != 0;
                        if (pre[u] && !want) actions[gi[u]] = 0.f;               /* main.py:401 */
                    }
                    bal[u] = __ballot_sync(0xffffffffu, want);
                    cnt += __popc(bal[u]);
                }
                int base = 0;
                if (lane == 0) {
                    const long long t0 = clock64();
                    while (*reinterpret_cast<volatile int *>(&C->q_res) + cnt + PVT_MARGIN - *reinterpret_cast<volatile int *>(&C->q_free) > PVT_RING) {
                        __nanosleep(100); PVT_TIMEOUT(t0);
                    }
                    base = atomicAdd(&C->q_res, cnt);
                }
                base = __shfl_sync(0xffffffffu, base, 0);
#pragma unroll
                for (int u = 0; u < PVT_PCHUNKS; ++u) {
                    if ((bal[u] >> lane) & 1u)
                        *reinterpret_cast<volatile int *>(&ring[(base + __popc(bal[u] & lt)) & (PVT_RING - 1)]) = gi[u] * slot_step;
                    base += __popc(bal[u]);
                }
            }
            first = false;
            if (!PVT_PREFETCH && lane == 0) ntk = dyn0 + atomicAdd(&ticket[0], PVT_BATCH);
            tk = __shfl_sync(0xffffffffu, ntk, 0);
        }
        __threadfence_block();
        __syncwarp();
        if (lane == 0 && atomicAdd(&C->p_done, 1) == PVT_PRODUCERS - 1) {
            __threadfence_block();
            *reinterpret_cast<volatile int *>(&C->q_done) = 1;
        }
    }
    pvt_teardown(tmem);
    if (tid == 0 && atomicAdd(&ticket[1], 1) == (int)gridDim.x - 1) { ticket[0] = 0; ticket[1] = 0; }
}

/* ---- critic: same contract as pve_critic_kernel (nstep.cuh) ------------------------------------------ */
template <int STRIDE>
__global__ void __launch_bounds__(PVT_THREADS_CRITIC, 1)
pve_critic_tc_kernel(const __grid_constant__ PvtVecs V, const uint16_t *__restrict__ PW, const float *__restrict__ obs,
                     const float *__restrict__ act7, float *__restrict__ q, const long long n_rows_max,
                     const int32_t *__restrict__ n_rows_dev) {
    extern __shared__ __align__(128) unsigned char pvt_smem[];
    const long long n_rows = n_rows_dev ? min(n_rows_max, (long long)n_rows_dev[0]) : n_rows_max;
    if ((long long)blockIdx.x * PVT_GROUPS * PVT_TILE >= n_rows) return;
    PvtCtrl *const C = reinterpret_cast<PvtCtrl *>(pvt_smem + PVT_W_BYTES + PVT_GROUPS * 3 * PVT_A_SPLIT(1));
    uint32_t tmem;
    PvtGroup G;
    pvt_setup<true>(pvt_smem, PW, C, G, tmem);
    const int g = (int)(threadIdx.x >> 7);
    for (long long t0 = ((long long)blockIdx.x * PVT_GROUPS + g) * PVT_TILE; t0 < n_rows; t0 += (long long)gridDim.x * PVT_GROUPS * PVT_TILE) {
        const long long row = t0 + G.gt;
        const bool valid = row < n_rows;
        const float o = pvt_round<true>(V, G, valid ? obs + row * STRIDE : nullptr, valid ? act7 + row * 7 : nullptr);
        if (valid) q[row] = o;                                                   /* NET:73 */
    }
    pvt_teardown(tmem);
}
#endif  /* __CUDACC__ */
#endif
