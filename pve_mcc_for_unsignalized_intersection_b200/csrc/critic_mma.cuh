/* Tensor-core version of the critic (model_agent_maddpg.py:52-76; see nstep.cuh for the CUDA-core version and
 * actor_mma.cuh for the scheme): both dense layers as bf16 x 3 split-precision products on
 * mma.sync.m16n8k16 with fp32 accumulation, which keeps the fp32 graph's accuracy (same test bound).
 *
 *     x  = LN(obs[r][0][0..27])                                            NET:58-59
 *     h1 = ReLU(LN(x W1 + b1))                    28 -> 64, 2 k-slices     NET:60-64
 *     h2 = ReLU(LN([h1, a_0 .. a_6] W2 + b2))     71 -> 64, 5 k-slices     NET:66-71
 *     q  = h2 w3 + b3                                                       NET:73
 *
 * A warp owns 16 agents.  As in the actor, the accumulator fragments of layer 1 are the A fragments of the first
 * four k-slices of layer 2; the fifth slice (k = 64 .. 79) carries the 7 actions in its first 7 columns: in the
 * m16k16 A fragment those are registers a0 (row g) and a1 (row g + 8), columns 2t, 2t + 1 -- loaded straight from
 * act7, no shared memory.  Persistent CTAs (8 warps = 128 agents per tile) stride over the agent rows; the row
 * count is read on the device.
 */
#ifndef PVE_CRITIC_MMA_CUH
#define PVE_CRITIC_MMA_CUH

#include "actor_mma.cuh"
#include "nstep.cuh"

/* packed parameter block (32-bit words) */
enum { PVQ_WF1 = 0,                                   /* [2 kk][8 j][3 split][32 lanes][2] bf16x2 */
       PVQ_WF2 = PVQ_WF1 + 2 * 8 * 3 * 64,            /* [5 kk][8 j][3 split][32 lanes][2] bf16x2 (rows 71..79 = 0) */
       PVQ_VEC = PVQ_WF2 + 5 * 8 * 3 * 64,
       PVQ_LN0_G = PVQ_VEC, PVQ_LN0_B = PVQ_LN0_G + 32, PVQ_B1 = PVQ_LN0_B + 32, PVQ_LN1_G = PVQ_B1 + 64,
       PVQ_LN1_B = PVQ_LN1_G + 64, PVQ_B2 = PVQ_LN1_B + 64, PVQ_LN2_G = PVQ_B2 + 64, PVQ_LN2_B = PVQ_LN2_G + 64,
       PVQ_W3 = PVQ_LN2_B + 64, PVQ_B3 = PVQ_W3 + 64, PVQ_WORDS = PVQ_B3 + 4 };

/* W: flat fp32 critic parameters in the order of include/pve_mcc.h; out: PVQ_WORDS 32-bit words */
static inline void pvq_pack(const float *W, uint32_t *out) {
    memset(out, 0, sizeof(uint32_t) * PVQ_WORDS);
    for (int layer = 0; layer < 2; ++layer) {
        const int K = layer ? 71 : 28, KK = layer ? 5 : 2;
        const float *Wm = W + (layer ? PVC_W2 : PVC_W1);               /* [K][64] row-major */
        uint32_t *dst = out + (layer ? PVQ_WF2 : PVQ_WF1);
        for (int kk = 0; kk < KK; ++kk)
            for (int j = 0; j < 8; ++j)
                for (int lane = 0; lane < 32; ++lane)
                    for (int reg = 0; reg < 2; ++reg) {
                        const int g = lane >> 2, t = lane & 3, n = 8 * j + g, k0 = 16 * kk + 2 * t + 8 * reg;
                        uint16_t e0[3] = {0, 0, 0}, e1[3] = {0, 0, 0};
                        if (k0 < K) pvm_split3(Wm[k0 * 64 + n], e0);
                        if (k0 + 1 < K) pvm_split3(Wm[(k0 + 1) * 64 + n], e1);
                        for (int s = 0; s < 3; ++s)
                            dst[(((kk * 8 + j) * 3 + s) * 32 + lane) * 2 + reg] = (uint32_t)e0[s] | ((uint32_t)e1[s] << 16);
                    }
    }
    float *v = (float *)out;
    memcpy(v + PVQ_LN0_G, W + PVC_LN0_G, 28 * 4); memcpy(v + PVQ_LN0_B, W + PVC_LN0_B, 28 * 4);
    memcpy(v + PVQ_B1, W + PVC_B1, 64 * 4); memcpy(v + PVQ_LN1_G, W + PVC_LN1_G, 64 * 4);
    memcpy(v + PVQ_LN1_B, W + PVC_LN1_B, 64 * 4); memcpy(v + PVQ_B2, W + PVC_B2, 64 * 4);
    memcpy(v + PVQ_LN2_G, W + PVC_LN2_G, 64 * 4); memcpy(v + PVQ_LN2_B, W + PVC_LN2_B, 64 * 4);
    memcpy(v + PVQ_W3, W + PVC_W3, 64 * 4); v[PVQ_B3] = W[PVC_B3];
}

#ifdef __CUDACC__
#define PVQ_THREADS 256
#define PVQ_TILE 128
#define PVQ_SMEM_BYTES (PVQ_WORDS * 4 + PVQ_TILE * PVM_AS * 4)

/* 16 agents of this warp: rows row0 + 16 warp .. + 15; STRIDE as in pvc_round */
template <int STRIDE>
__device__ __forceinline__ void pvq_warp_round(const uint32_t *__restrict__ pw, float *__restrict__ a, const long long row0,
                                               const int n_valid, const float *__restrict__ obs,
                                               const float *__restrict__ act7, float *__restrict__ q) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
    const float *vec = reinterpret_cast<const float *>(pw);
    float *aw = a + warp * 16 * PVM_AS;
    /* first LayerNorm (NET:58-59): lanes l and l + 16 share row l (float4 pieces 0-3 / 4-6) */
    {
        const int r = lane & 15, half = lane >> 4, row = warp * 16 + r;
        const bool valid = row < n_valid;
        const float4 *src = reinterpret_cast<const float4 *>(obs + (row0 + (valid ? row : 0)) * STRIDE) + half * 4;
        float4 x[4];
#pragma unroll
        for (int p = 0; p < 4; ++p)
            x[p] = (valid && half * 4 + p < 7) ? src[p] : make_float4(0.f, 0.f, 0.f, 0.f);
        float s = ((x[0].x + x[0].y) + (x[0].z + x[0].w)) + ((x[1].x + x[1].y) + (x[1].z + x[1].w))
                  + ((x[2].x + x[2].y) + (x[2].z + x[2].w)) + ((x[3].x + x[3].y) + (x[3].z + x[3].w));
        s += __shfl_xor_sync(0xffffffffu, s, 16);
        const float mean = s * (1.f / 28.f);
        float q2 = 0.f;
#pragma unroll
        for (int p = 0; p < 4; ++p)
            if (half * 4 + p < 7) {
                const float d0 = x[p].x - mean, d1 = x[p].y - mean, d2 = x[p].z - mean, d3 = x[p].w - mean;
                q2 = fmaf(d0, d0, q2); q2 = fmaf(d1, d1, q2); q2 = fmaf(d2, d2, q2); q2 = fmaf(d3, d3, q2);
            }
        q2 += __shfl_xor_sync(0xffffffffu, q2, 16);
        const float rs = rsqrtf(q2 * (1.f / 28.f) + PVA_EPS);
#pragma unroll
        for (int p = 0; p < 4; ++p) {
            const int c = (half * 4 + p) * 4;                    /* columns 28..31 come out as 0 (gamma = beta = 0) */
            const float4 gm = *reinterpret_cast<const float4 *>(vec + PVQ_LN0_G + c);
            const float4 bt = *reinterpret_cast<const float4 *>(vec + PVQ_LN0_B + c);
            const float i0 = rs * gm.x, i1 = rs * gm.y, i2 = rs * gm.z, i3 = rs * gm.w;
            float4 y;
            y.x = fmaf(x[p].x, i0, fmaf(-mean, i0, bt.x)); y.y = fmaf(x[p].y, i1, fmaf(-mean, i1, bt.y));
            y.z = fmaf(x[p].z, i2, fmaf(-mean, i2, bt.z)); y.w = fmaf(x[p].w, i3, fmaf(-mean, i3, bt.w));
            *reinterpret_cast<float4 *>(aw + r * PVM_AS + c) = y;
        }
    }
    /* the action columns of this lane: rows g and g + 8, columns 2t and 2t + 1 (column 7 is padding) */
    float a00 = 0.f, a01 = 0.f, a10 = 0.f, a11 = 0.f;
    {
        const int rg = warp * 16 + g;
        if (rg < n_valid) { a00 = act7[(row0 + rg) * 7 + 2 * t]; if (t < 3) a01 = act7[(row0 + rg) * 7 + 2 * t + 1]; }
        if (rg + 8 < n_valid) { a10 = act7[(row0 + rg + 8) * 7 + 2 * t]; if (t < 3) a11 = act7[(row0 + rg + 8) * 7 + 2 * t + 1]; }
    }
    __syncwarp();
    float acc[8][4];
#pragma unroll
    for (int j = 0; j < 8; ++j) { acc[j][0] = 0.f; acc[j][1] = 0.f; acc[j][2] = 0.f; acc[j][3] = 0.f; }
    /* Dense 28 -> 64 (NET:60): A fragments from the tile */
#pragma unroll
    for (int kk = 0; kk < 2; ++kk) {
        const float2 v00 = *reinterpret_cast<const float2 *>(aw + g * PVM_AS + 16 * kk + 2 * t);
        const float2 v10 = *reinterpret_cast<const float2 *>(aw + (g + 8) * PVM_AS + 16 * kk + 2 * t);
        const float2 v01 = *reinterpret_cast<const float2 *>(aw + g * PVM_AS + 16 * kk + 8 + 2 * t);
        const float2 v11 = *reinterpret_cast<const float2 *>(aw + (g + 8) * PVM_AS + 16 * kk + 8 + 2 * t);
        uint32_t ah[4], am[4], al[4];
        pvm_split_pair(v00.x, v00.y, ah[0], am[0], al[0]);
        pvm_split_pair(v10.x, v10.y, ah[1], am[1], al[1]);
        pvm_split_pair(v01.x, v01.y, ah[2], am[2], al[2]);
        pvm_split_pair(v11.x, v11.y, ah[3], am[3], al[3]);
        pvm_kstep(acc, ah, am, al, pw + PVQ_WF1, kk, lane);
    }
    __syncwarp();                                                /* the tile rows may be overwritten next round */
    pvm_ln_relu(acc, vec + PVQ_B1, vec + PVQ_LN1_G, vec + PVQ_LN1_B, t);             /* NET:60-64 */
    /* Dense 71 -> 64 (NET:66-67): four slices from the accumulators, the fifth from the actions */
    float acc2[8][4];
#pragma unroll
    for (int j = 0; j < 8; ++j) { acc2[j][0] = 0.f; acc2[j][1] = 0.f; acc2[j][2] = 0.f; acc2[j][3] = 0.f; }
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
        uint32_t ah[4], am[4], al[4];
        pvm_split_pair(acc[2 * kk][0], acc[2 * kk][1], ah[0], am[0], al[0]);
        pvm_split_pair(acc[2 * kk][2], acc[2 * kk][3], ah[1], am[1], al[1]);
        pvm_split_pair(acc[2 * kk + 1][0], acc[2 * kk + 1][1], ah[2], am[2], al[2]);
        pvm_split_pair(acc[2 * kk + 1][2], acc[2 * kk + 1][3], ah[3], am[3], al[3]);
        pvm_kstep(acc2, ah, am, al, pw + PVQ_WF2, kk, lane);
    }
    {
        uint32_t ah[4], am[4], al[4];
        pvm_split_pair(a00, a01, ah[0], am[0], al[0]);
        pvm_split_pair(a10, a11, ah[1], am[1], al[1]);
        ah[2] = am[2] = al[2] = 0u; ah[3] = am[3] = al[3] = 0u;   /* columns 72..79 */
        pvm_kstep(acc2, ah, am, al, pw + PVQ_WF2, 4, lane);
    }
    pvm_ln_relu(acc2, vec + PVQ_B2, vec + PVQ_LN2_G, vec + PVQ_LN2_B, t);            /* NET:67-71 */
    /* Dense 64 -> 1 (NET:73) */
    float o0 = 0.f, o1 = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float2 u = *reinterpret_cast<const float2 *>(vec + PVQ_W3 + 8 * j + 2 * t);
        o0 = fmaf(acc2[j][0], u.x, o0); o0 = fmaf(acc2[j][1], u.y, o0);
        o1 = fmaf(acc2[j][2], u.x, o1); o1 = fmaf(acc2[j][3], u.y, o1);
    }
    o0 += __shfl_xor_sync(0xffffffffu, o0, 1); o1 += __shfl_xor_sync(0xffffffffu, o1, 1);
    o0 += __shfl_xor_sync(0xffffffffu, o0, 2); o1 += __shfl_xor_sync(0xffffffffu, o1, 2);
    if (t < 2) {                                                 /* lane t = 0 writes row g, t = 1 row g + 8 */
        const int row = warp * 16 + g + 8 * t;
        if (row < n_valid) q[row0 + row] = (t ? o1 : o0) + vec[PVQ_B3];
    }
}

/* same contract as pve_critic_kernel (nstep.cuh); PW = the packed block of pvq_pack */
template <int STRIDE>
__global__ void __launch_bounds__(PVQ_THREADS, 2)
pve_critic_mma_kernel(const uint32_t *__restrict__ PW, const float *__restrict__ obs, const float *__restrict__ act7,
                      float *__restrict__ q, const long long n_rows_max, const int32_t *__restrict__ n_rows_dev) {
    extern __shared__ __align__(16) unsigned char pvq_smem[];
    uint32_t *const pw = reinterpret_cast<uint32_t *>(pvq_smem);
    float *const a = reinterpret_cast<float *>(pw + PVQ_WORDS);
    const long long n_rows = n_rows_dev ? min(n_rows_max, (long long)n_rows_dev[0]) : n_rows_max;
    if ((long long)blockIdx.x * PVQ_TILE >= n_rows) return;
    for (int i = threadIdx.x; i < PVQ_WORDS / 4; i += PVQ_THREADS)
        reinterpret_cast<uint4 *>(pw)[i] = reinterpret_cast<const uint4 *>(PW)[i];
    __syncthreads();
    for (long long t0 = (long long)blockIdx.x * PVQ_TILE; t0 < n_rows; t0 += (long long)gridDim.x * PVQ_TILE) {
        const int n_valid = (int)min((long long)PVQ_TILE, n_rows - t0);
        if ((int)(threadIdx.x >> 5) * 16 < n_valid) pvq_warp_round<STRIDE>(pw, a, t0, n_valid, obs, act7, q);
    }
}
#endif  /* __CUDACC__ */
#endif
