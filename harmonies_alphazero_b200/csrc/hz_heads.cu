// hz_heads.cu — fused policy/value heads of the reference network (model.py:340-355) for the
// batched leaf evaluation: ONE kernel instead of ~10 library launches per simulation step.
//
//   x      [n, 35, C]  bf16, NHWC output of the residual tower (C = cnn_filters)
//   glob   [n, 42]     bf16 global features
//   -> 1x1 convs (2 policy + 1 value channel, BatchNorm folded) + ReLU          (model.py:340-343,349-351)
//   -> policy: flatten (channel-major, as .view on NCHW) ++ glob -> FC 112->143  (:344-347)
//   -> value : flatten ++ glob -> FC 77->H -> ReLU -> FC H->1 -> tanh            (:352-355)
//   logits [n,143] fp32, value [n] fp32.  All accumulation in fp32.
//
// The tower stays cuDNN (north_star: "the network stays PyTorch"); this tail is ~0.1 MFLOP
// and 9 KB of reads per position, i.e. HBM/launch-bound glue that is cheaper fused.
// Mapping: a block of 256 threads takes 7 positions at a time: thread = (position, cell) for
// the 1x1 convs, then thread = output unit for the FC layers with the 7 positions held as 7
// accumulators, so each weight is read once per 7 positions (weights stay in L1/L2).
#include <math.h>

#include "hz_common.cuh"

namespace hz {

constexpr int HP = 7;          // positions per block iteration (7*35 = 245 <= 256 threads)
constexpr int HTPB = 256;
constexpr int CELLS = 35;
constexpr int NGLOB = 42;
constexpr int NPOL = 143;
constexpr int PIN = 2 * CELLS + NGLOB;   // 112
constexpr int VIN = CELLS + NGLOB;       // 77

struct HeadParams {
    const float* w_conv;   // [3][C]   rows: policy ch0, policy ch1, value ch0
    const float* b_conv;   // [3]
    const float* w_pol_t;  // [112][143]  transposed policy_fc weight
    const float* b_pol;    // [143]
    const float* w_v1_t;   // [77][H]     transposed value_fc1 weight
    const float* b_v1;     // [H]
    const float* w_v2;     // [H]
    float b_v2;
    int C, H;
};

__global__ void __launch_bounds__(HTPB) k_heads(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ glob,
                                                int64_t n, HeadParams P, float* __restrict__ logits,
                                                float* __restrict__ value) {
    extern __shared__ __align__(16) float smem[];
    float* s_wc = smem;                         // [3][C]
    float* s_pin = s_wc + 3 * P.C;              // [HP][112]  policy FC input per position
    float* s_vin = s_pin + HP * PIN;            // [HP][80]   value FC input per position (77 used)
    float* s_red = s_vin + HP * 80;             // [HP][8]    per-warp partial sums of the last FC
    for (int i = threadIdx.x; i < 3 * P.C; i += HTPB) s_wc[i] = P.w_conv[i];
    const float bc0 = P.b_conv[0], bc1 = P.b_conv[1], bc2 = P.b_conv[2];
    const int C = P.C, H = P.H;
    int64_t n_groups = (n + HP - 1) / HP;
    for (int64_t grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
        int64_t base = grp * HP;
        int cnt = (int)min((int64_t)HP, n - base);
        __syncthreads();
        // ---- 1x1 convs + ReLU: thread = (position, cell); one contiguous C-row of bf16 each
        int t = threadIdx.x;
        if (t < cnt * CELLS) {
            int p = t / CELLS, cell = t - CELLS * p;
            const uint4* row = reinterpret_cast<const uint4*>(x + ((base + p) * CELLS + cell) * (int64_t)C);
            float a0 = bc0, a1 = bc1, a2 = bc2;
            const float4* w0 = reinterpret_cast<const float4*>(s_wc);
            const float4* w1 = reinterpret_cast<const float4*>(s_wc + C);
            const float4* w2 = reinterpret_cast<const float4*>(s_wc + 2 * C);
#pragma unroll 4
            for (int v = 0; v < C / 8; v++) {
                uint4 q = row[v];
                const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&q);
                float2 f0 = __bfloat1622float2(h[0]), f1 = __bfloat1622float2(h[1]);
                float2 f2 = __bfloat1622float2(h[2]), f3 = __bfloat1622float2(h[3]);
                // explicit fmaf: the library is built with --fmad=false for the search arithmetic
#define HZ_DOT8(acc, W)                                                                              \
                { float4 wa = W[2 * v], wb = W[2 * v + 1];                                               \
                  acc = fmaf(f0.x, wa.x, acc); acc = fmaf(f0.y, wa.y, acc); acc = fmaf(f1.x, wa.z, acc); \
                  acc = fmaf(f1.y, wa.w, acc); acc = fmaf(f2.x, wb.x, acc); acc = fmaf(f2.y, wb.y, acc); \
                  acc = fmaf(f3.x, wb.z, acc); acc = fmaf(f3.y, wb.w, acc); }
                HZ_DOT8(a0, w0) HZ_DOT8(a1, w1) HZ_DOT8(a2, w2)
#undef HZ_DOT8
            }
            s_pin[p * PIN + cell] = fmaxf(a0, 0.0f);            // channel-major flatten (model.py:343)
            s_pin[p * PIN + CELLS + cell] = fmaxf(a1, 0.0f);
            s_vin[p * 80 + cell] = fmaxf(a2, 0.0f);
        }
        for (int i = threadIdx.x; i < cnt * NGLOB; i += HTPB) {   // ++ global features (:344-346,352)
            int p = i / NGLOB, g = i - NGLOB * p;
            float gv = __bfloat162float(glob[(base + p) * NGLOB + g]);
            s_pin[p * PIN + 2 * CELLS + g] = gv;
            s_vin[p * 80 + CELLS + g] = gv;
        }
        __syncthreads();
        // The two FC stacks run side by side: warps 0-2 the policy FC, warps 3-7 the value FCs.
        // Each thread owns TWO output units x 7 positions (14 accumulators) and reads the
        // inputs as float4 along j, so an inner step is 7 LDS.128 + 8 LDG + 56 FMA.
        float part[HP];
#pragma unroll
        for (int p = 0; p < HP; p++) part[p] = 0.0f;
        if (t < 96) {
            // ---- policy FC 112 -> 143 (model.py:344-347)
            if (t < 72) {
                int a0i = t, a1i = t + 72;
                bool has1 = a1i < NPOL;
                int a1c = has1 ? a1i : a0i;
                float acc0[HP], acc1[HP];
#pragma unroll
                for (int p = 0; p < HP; p++) { acc0[p] = P.b_pol[a0i]; acc1[p] = P.b_pol[a1c]; }
#pragma unroll 2
                for (int j = 0; j < PIN; j += 4) {
                    float wa[4], wb[4];
#pragma unroll
                    for (int k = 0; k < 4; k++) { wa[k] = __ldg(P.w_pol_t + (j + k) * NPOL + a0i); wb[k] = __ldg(P.w_pol_t + (j + k) * NPOL + a1c); }
#pragma unroll
                    for (int p = 0; p < HP; p++) {
                        float4 in = *reinterpret_cast<const float4*>(s_pin + p * PIN + j);
                        acc0[p] = fmaf(wa[0], in.x, acc0[p]); acc0[p] = fmaf(wa[1], in.y, acc0[p]);
                        acc0[p] = fmaf(wa[2], in.z, acc0[p]); acc0[p] = fmaf(wa[3], in.w, acc0[p]);
                        acc1[p] = fmaf(wb[0], in.x, acc1[p]); acc1[p] = fmaf(wb[1], in.y, acc1[p]);
                        acc1[p] = fmaf(wb[2], in.z, acc1[p]); acc1[p] = fmaf(wb[3], in.w, acc1[p]);
                    }
                }
#pragma unroll
                for (int p = 0; p < HP; p++) {
                    if (p < cnt) {
                        logits[(base + p) * NPOL + a0i] = acc0[p];
                        if (has1) logits[(base + p) * NPOL + a1i] = acc1[p];
                    }
                }
            }
        } else {
            // ---- value FC 77 -> H -> ReLU -> dot w2 (model.py:352-354): units u and u + H/2
            int half = H / 2;
            for (int u = t - 96; u < half; u += HTPB - 96) {
                int u1 = u + half;
                float acc0[HP], acc1[HP];
#pragma unroll
                for (int p = 0; p < HP; p++) { acc0[p] = P.b_v1[u]; acc1[p] = P.b_v1[u1]; }
#pragma unroll 2
                for (int j = 0; j < 76; j += 4) {
                    float wa[4], wb[4];
#pragma unroll
                    for (int k = 0; k < 4; k++) { wa[k] = __ldg(P.w_v1_t + (j + k) * H + u); wb[k] = __ldg(P.w_v1_t + (j + k) * H + u1); }
#pragma unroll
                    for (int p = 0; p < HP; p++) {
                        float4 in = *reinterpret_cast<const float4*>(s_vin + p * 80 + j);
                        acc0[p] = fmaf(wa[0], in.x, acc0[p]); acc0[p] = fmaf(wa[1], in.y, acc0[p]);
                        acc0[p] = fmaf(wa[2], in.z, acc0[p]); acc0[p] = fmaf(wa[3], in.w, acc0[p]);
                        acc1[p] = fmaf(wb[0], in.x, acc1[p]); acc1[p] = fmaf(wb[1], in.y, acc1[p]);
                        acc1[p] = fmaf(wb[2], in.z, acc1[p]); acc1[p] = fmaf(wb[3], in.w, acc1[p]);
                    }
                }
                {   // j = 76 (VIN = 77)
                    float wa = __ldg(P.w_v1_t + 76 * H + u), wb = __ldg(P.w_v1_t + 76 * H + u1);
#pragma unroll
                    for (int p = 0; p < HP; p++) {
                        float in = s_vin[p * 80 + 76];
                        acc0[p] = fmaf(wa, in, acc0[p]); acc1[p] = fmaf(wb, in, acc1[p]);
                    }
                }
                float w2a = P.w_v2[u], w2b = P.w_v2[u1];
#pragma unroll
                for (int p = 0; p < HP; p++) {
                    part[p] = fmaf(fmaxf(acc0[p], 0.0f), w2a, part[p]);
                    part[p] = fmaf(fmaxf(acc1[p], 0.0f), w2b, part[p]);
                }
            }
        }
#pragma unroll
        for (int p = 0; p < HP; p++) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) part[p] += __shfl_xor_sync(0xFFFFFFFFu, part[p], o);
        }
        if ((t & 31) == 0) {
#pragma unroll
            for (int p = 0; p < HP; p++) s_red[p * 8 + (t >> 5)] = part[p];
        }
        __syncthreads();
        if (t < cnt) {
            float s = P.b_v2;
#pragma unroll
            for (int w = 0; w < HTPB / 32; w++) s += s_red[t * 8 + w];
            value[base + t] = tanhf(s);                         // model.py:355
        }
    }
}

// ---- the default network's shape (C = 128, H = 256): persistent variant ----------------------
// One 512-thread block per SM keeps BOTH FC weight matrices in shared memory (143 KB fp32, read
// from L2 once per block instead of once per 7 positions) and walks groups of 14 positions:
//   phase 1  the 1x1 convs as [cells x 128] x [128 x 3] on the tensor cores: a warp takes 16 board
//            cells per mma.sync m16n8k16 tile; A fragments are the bf16 activations loaded straight
//            from global memory with 16-byte requests (the K order is permuted so that a lane's
//            uint4 IS its fragment), B = the conv weights split into bf16 hi + lo parts held in
//            registers (two MMAs per k-step: fp32-weight accuracy, 2^-17 relative)
//   phase 2  thread = 2 output units x 7 positions (14 accumulators): per 4 inputs 8 weight
//            words + 7 broadcast LDS.128 feed 56 FMAs
constexpr int FG = 14;
constexpr int FTPB = 512;
constexpr int FC = 128, FH = 256;
constexpr int WPN = PIN * NPOL + 16;     // policy weights, flat copy of w_pol_t (+ slack: unit "143" reads are discarded)
constexpr size_t FSMEM = sizeof(float) * (size_t)(WPN + 77 * FH + FG * PIN + FG * 80 + FG * 4);

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void mma_bf16_16816(float c[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3,
                                               uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_bf16(__nv_bfloat16 lo, __nv_bfloat16 hi) {
    return (uint32_t)__bfloat16_as_ushort(lo) | ((uint32_t)__bfloat16_as_ushort(hi) << 16);
}

__global__ void __launch_bounds__(FTPB, 1) k_heads_p(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ glob,
                                                     int64_t n, HeadParams P, float* __restrict__ logits,
                                                     float* __restrict__ value) {
    extern __shared__ __align__(16) float smem[];
    float* s_wp = smem;                      // [112][143] (+ slack)
    float* s_wv = s_wp + WPN;                // [77][256]
    float* s_pin = s_wv + 77 * FH;           // [FG][112]
    float* s_vin = s_pin + FG * PIN;         // [FG][80]
    float* s_red = s_vin + FG * 80;          // [FG][4]
    const int t = threadIdx.x, warp = t >> 5, g8 = (t & 31) >> 2, q4 = t & 3;
    // FC weights -> shared memory, asynchronously: phase 1 of the first group does not need them
    for (int i = t; i < PIN * NPOL / 4; i += FTPB) cp_async16(s_wp + 4 * i, P.w_pol_t + 4 * i);
    for (int i = t; i < 77 * FH / 4; i += FTPB) cp_async16(s_wv + 4 * i, P.w_v1_t + 4 * i);
    asm volatile("cp.async.commit_group;" ::: "memory");
    if (t < 16) s_wp[PIN * NPOL + t] = 0.0f;
    // B fragments of the conv weights: output n = g8 (0,1 policy, 2 value, others zero); the lane's
    // k rows of k-step ks = (kk, s) are channels 32 kk + 8 q4 + 4 s + {0,1} and + {2,3}
    uint32_t bh[16], bl[16];
#pragma unroll
    for (int ks = 0; ks < 8; ks++) {
#pragma unroll
        for (int w = 0; w < 2; w++) {
            int ch = 32 * (ks >> 1) + 8 * q4 + 4 * (ks & 1) + 2 * w;
            const bool live = g8 < 3;
            float w0 = live ? P.w_conv[g8 * FC + ch] : 0.0f, w1 = live ? P.w_conv[g8 * FC + ch + 1] : 0.0f;
            __nv_bfloat16 h0 = __float2bfloat16_rn(w0), h1 = __float2bfloat16_rn(w1);
            bh[ks * 2 + w] = pack_bf16(h0, h1);
            bl[ks * 2 + w] = pack_bf16(__float2bfloat16_rn(w0 - __bfloat162float(h0)), __float2bfloat16_rn(w1 - __bfloat162float(h1)));
        }
    }
    const float bc0 = P.b_conv[0], bc1 = P.b_conv[1], bc2 = P.b_conv[2];
    int64_t n_groups = (n + FG - 1) / FG;
    bool weights_pending = true;
    for (int64_t grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
        int64_t base = grp * FG;
        int cnt = (int)min((int64_t)FG, n - base), ncell = cnt * CELLS;
        __syncthreads();
        // ---- phase 1: 1x1 convs + ReLU (model.py:340-343,349-351)
        const uint4* rows = reinterpret_cast<const uint4*>(x + base * CELLS * (int64_t)FC);
        for (int tile = warp; tile * 16 < ncell; tile += FTPB / 32) {
            int r0 = tile * 16 + g8, r1 = r0 + 8;
            uint4 qa[4], qb[4];
#pragma unroll
            for (int kk = 0; kk < 4; kk++) {
                qa[kk] = r0 < ncell ? rows[r0 * (FC / 8) + kk * 4 + q4] : make_uint4(0, 0, 0, 0);
                qb[kk] = r1 < ncell ? rows[r1 * (FC / 8) + kk * 4 + q4] : make_uint4(0, 0, 0, 0);
            }
            float c[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
            for (int kk = 0; kk < 4; kk++) {
                mma_bf16_16816(c, qa[kk].x, qb[kk].x, qa[kk].y, qb[kk].y, bh[kk * 4], bh[kk * 4 + 1]);
                mma_bf16_16816(c, qa[kk].x, qb[kk].x, qa[kk].y, qb[kk].y, bl[kk * 4], bl[kk * 4 + 1]);
                mma_bf16_16816(c, qa[kk].z, qb[kk].z, qa[kk].w, qb[kk].w, bh[kk * 4 + 2], bh[kk * 4 + 3]);
                mma_bf16_16816(c, qa[kk].z, qb[kk].z, qa[kk].w, qb[kk].w, bl[kk * 4 + 2], bl[kk * 4 + 3]);
            }
            // c[0], c[1] = row r0, outputs 2 q4, 2 q4 + 1;  c[2], c[3] = row r1
            if (q4 < 2) {
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    int r = h ? r1 : r0;
                    if (r < ncell) {
                        int p = r / CELLS, cell = r - CELLS * p;
                        if (q4 == 0) {
                            s_pin[p * PIN + cell] = fmaxf(c[2 * h] + bc0, 0.0f);          // channel-major flatten (model.py:343)
                            s_pin[p * PIN + CELLS + cell] = fmaxf(c[2 * h + 1] + bc1, 0.0f);
                        } else {
                            s_vin[p * 80 + cell] = fmaxf(c[2 * h] + bc2, 0.0f);
                        }
                    }
                }
            }
        }
        for (int i = t; i < cnt * NGLOB; i += FTPB) {   // ++ global features (:344-346,352)
            int p = i / NGLOB, g = i - NGLOB * p;
            float gv = __bfloat162float(glob[(base + p) * NGLOB + g]);
            s_pin[p * PIN + 2 * CELLS + g] = gv;
            s_vin[p * 80 + CELLS + g] = gv;
        }
        if (weights_pending) {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            weights_pending = false;
        }
        __syncthreads();
        // ---- phase 2: warps 0-5 policy FC (two halves of 7 positions), warps 6-13 value FCs
        if (t < 192) {
            int half = t / 96, u0 = t - 96 * half;
            if (u0 < 72) {
                int u1 = u0 + 72, p0 = half * 7;            // u1 == 143 (thread 71) reads a neighbour's weights; never stored
                float acc0[7], acc1[7];
                float b0 = P.b_pol[u0], b1 = u1 < NPOL ? P.b_pol[u1] : 0.0f;
#pragma unroll
                for (int p = 0; p < 7; p++) { acc0[p] = b0; acc1[p] = b1; }
#pragma unroll 2
                for (int j = 0; j < PIN; j += 4) {
                    float wa[4], wb[4];
#pragma unroll
                    for (int k = 0; k < 4; k++) { wa[k] = s_wp[(j + k) * NPOL + u0]; wb[k] = s_wp[(j + k) * NPOL + u1]; }
#pragma unroll
                    for (int p = 0; p < 7; p++) {
                        float4 in = *reinterpret_cast<const float4*>(s_pin + (p0 + p) * PIN + j);
                        acc0[p] = fmaf(wa[0], in.x, acc0[p]); acc0[p] = fmaf(wa[1], in.y, acc0[p]);
                        acc0[p] = fmaf(wa[2], in.z, acc0[p]); acc0[p] = fmaf(wa[3], in.w, acc0[p]);
                        acc1[p] = fmaf(wb[0], in.x, acc1[p]); acc1[p] = fmaf(wb[1], in.y, acc1[p]);
                        acc1[p] = fmaf(wb[2], in.z, acc1[p]); acc1[p] = fmaf(wb[3], in.w, acc1[p]);
                    }
                }
#pragma unroll
                for (int p = 0; p < 7; p++) {
                    if (p0 + p < cnt) {
                        logits[(base + p0 + p) * NPOL + u0] = acc0[p];
                        if (u1 < NPOL) logits[(base + p0 + p) * NPOL + u1] = acc1[p];
                    }
                }
            }
        } else if (t < 448) {
            int v = t - 192, half = v >> 7, u0 = v & 127, u1 = u0 + 128, p0 = half * 7;
            float acc0[7], acc1[7];
            float b0 = P.b_v1[u0], b1 = P.b_v1[u1];
#pragma unroll
            for (int p = 0; p < 7; p++) { acc0[p] = b0; acc1[p] = b1; }
#pragma unroll 2
            for (int j = 0; j < 76; j += 4) {
                float wa[4], wb[4];
#pragma unroll
                for (int k = 0; k < 4; k++) { wa[k] = s_wv[(j + k) * FH + u0]; wb[k] = s_wv[(j + k) * FH + u1]; }
#pragma unroll
                for (int p = 0; p < 7; p++) {
                    float4 in = *reinterpret_cast<const float4*>(s_vin + (p0 + p) * 80 + j);
                    acc0[p] = fmaf(wa[0], in.x, acc0[p]); acc0[p] = fmaf(wa[1], in.y, acc0[p]);
                    acc0[p] = fmaf(wa[2], in.z, acc0[p]); acc0[p] = fmaf(wa[3], in.w, acc0[p]);
                    acc1[p] = fmaf(wb[0], in.x, acc1[p]); acc1[p] = fmaf(wb[1], in.y, acc1[p]);
                    acc1[p] = fmaf(wb[2], in.z, acc1[p]); acc1[p] = fmaf(wb[3], in.w, acc1[p]);
                }
            }
            {   // j = 76 (VIN = 77)
                float wa = s_wv[76 * FH + u0], wb = s_wv[76 * FH + u1];
#pragma unroll
                for (int p = 0; p < 7; p++) {
                    float in = s_vin[(p0 + p) * 80 + 76];
                    acc0[p] = fmaf(wa, in, acc0[p]); acc1[p] = fmaf(wb, in, acc1[p]);
                }
            }
            float w2a = P.w_v2[u0], w2b = P.w_v2[u1];
#pragma unroll
            for (int p = 0; p < 7; p++) {
                float part = fmaf(fmaxf(acc1[p], 0.0f), w2b, fmaxf(acc0[p], 0.0f) * w2a);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xFFFFFFFFu, part, o);
                if ((t & 31) == 0) s_red[(p0 + p) * 4 + (u0 >> 5)] = part;
            }
        }
        __syncthreads();
        if (t < cnt) {
            float sum = P.b_v2 + s_red[t * 4] + s_red[t * 4 + 1] + s_red[t * 4 + 2] + s_red[t * 4 + 3];
            value[base + t] = tanhf(sum);                           // model.py:355
        }
    }
}

// ---- FC heads on the tensor cores (the tile path) --------------------------------------------------
// policy_fc (112 -> 143) and value_fc1 (77 -> 256) + value_fc2 + tanh for 32 positions per block, as mma.sync
// m16n8k16: M = 16 output units, N = 8 positions, K = 16 inputs.  Weights AND inputs are split into bf16 high + low
// parts and three products are accumulated in fp32 (hi*hi + hi*lo + lo*hi: 2^-16 relative, fp32-weight accuracy).
// A warp owns output-unit tiles; it reads its weight fragments straight from global memory (L2) into registers ONCE
// and reuses them for the block's four position tiles, so the 143 KB of weights are never staged in shared memory and
// there is a single block barrier before the arithmetic (the FMA kernel above, measured on this path, spent most of its 21 us at barriers).
constexpr int MB = 32;                        // positions per block
constexpr int MT_POL = 9, MT_VAL = 16;        // 16-unit tiles: 144 >= 143 policy logits, 256 hidden units
constexpr int KS_POL = 7, KS_VAL = 5;         // 16-input steps: 112, 80 >= 77
constexpr int SP = 120, SV = 88;              // shared-memory row strides in bf16 (bank-conflict free for the B fragments)
constexpr int MTPB = 512;
__device__ __forceinline__ void split_bf16(float v, __nv_bfloat16& hi, __nv_bfloat16& lo) {
    hi = __float2bfloat16_rn(v);
    lo = __float2bfloat16_rn(v - __bfloat162float(hi));
}
__global__ void __launch_bounds__(MTPB, 1) k_heads_fc_mma(const float* __restrict__ hc, const __nv_bfloat16* __restrict__ glob, int64_t n,
                                                          HeadParams P, float* __restrict__ logits, float* __restrict__ value,
                                                          const int* __restrict__ n_active) {
    __shared__ __align__(16) __nv_bfloat16 s_ph[MB][SP], s_pl[MB][SP], s_vh[MB][SV], s_vl[MB][SV];
    __shared__ float s_part[MT_VAL][MB];       // value_fc2 partial sums per unit tile: summed in a fixed order (bit-reproducible)
    if (n_active) n = min(n, (int64_t)max(*n_active, 0));
    const int64_t base = (int64_t)blockIdx.x * MB;
    if (base >= n) return;
    const int cnt = (int)min((int64_t)MB, n - base), t = threadIdx.x;
    // hc: what the tower's head item writes, [tile of 16 boards][filter * 35 + cell][board in tile]
    auto hc_at = [&](int64_t bd, int j) { return hc[(bd >> 4) * (3 * CELLS * 16) + j * 16 + (bd & 15)]; };
    // inputs (model.py:343-346,351-352): policy = [conv ch0 | conv ch1 | global], value = [conv ch2 | global], as bf16 hi + lo
    for (int i = t; i < MB * PIN; i += MTPB) {
        const int p = i / PIN, j = i - PIN * p;
        float v = 0.0f;
        if (p < cnt) v = j < 2 * CELLS ? hc_at(base + p, j) : __bfloat162float(glob[(base + p) * NGLOB + (j - 2 * CELLS)]);
        split_bf16(v, s_ph[p][j], s_pl[p][j]);
    }
    for (int i = t; i < MB * 80; i += MTPB) {
        const int p = i / 80, j = i - 80 * p;
        float v = 0.0f;
        if (p < cnt && j < VIN) v = j < CELLS ? hc_at(base + p, 2 * CELLS + j) : __bfloat162float(glob[(base + p) * NGLOB + (j - CELLS)]);
        split_bf16(v, s_vh[p][j], s_vl[p][j]);
    }
    for (int i = t; i < MT_VAL * MB; i += MTPB) (&s_part[0][0])[i] = 0.0f;
    __syncthreads();
    const int warp = t >> 5, lane = t & 31, g = lane >> 2, q = lane & 3;
    for (int mt = warp; mt < MT_POL + MT_VAL; mt += MTPB / 32) {
        const bool pol = mt < MT_POL;
        const int m = pol ? mt : mt - MT_POL, KS = pol ? KS_POL : KS_VAL, NU = pol ? NPOL : FH, KR = pol ? PIN : VIN;
        const float* __restrict__ WT = pol ? P.w_pol_t : P.w_v1_t;          // [input j][unit u]
        const int u0 = m * 16 + g, u1 = u0 + 8;
        uint32_t ah[KS_POL][4], al[KS_POL][4];
#pragma unroll
        for (int ks = 0; ks < KS_POL; ks++) {
            if (ks < KS) {
#pragma unroll
                for (int r = 0; r < 4; r++) {
                    const int u = (r & 1) ? u1 : u0, j = ks * 16 + 2 * q + (r >> 1) * 8;
                    const float w0 = (u < NU && j < KR) ? WT[(size_t)j * NU + u] : 0.0f;
                    const float w1 = (u < NU && j + 1 < KR) ? WT[(size_t)(j + 1) * NU + u] : 0.0f;
                    __nv_bfloat16 h0, l0, h1, l1;
                    split_bf16(w0, h0, l0);
                    split_bf16(w1, h1, l1);
                    ah[ks][r] = pack_bf16(h0, h1);
                    al[ks][r] = pack_bf16(l0, l1);
                }
            }
        }
        const float* __restrict__ B = pol ? P.b_pol : P.b_v1;
        const float bias0 = u0 < NU ? B[u0] : 0.0f, bias1 = u1 < NU ? B[u1] : 0.0f;
        const float w2a = (!pol) ? P.w_v2[u0] : 0.0f, w2b = (!pol) ? P.w_v2[u1] : 0.0f;
#pragma unroll 1
        for (int nt = 0; nt < MB / 8; nt++) {
            if (nt * 8 >= cnt) break;
            float c[4] = {bias0, bias0, bias1, bias1};
            const int p = nt * 8 + g;
            const __nv_bfloat16* rh = pol ? &s_ph[p][0] : &s_vh[p][0];
            const __nv_bfloat16* rl = pol ? &s_pl[p][0] : &s_vl[p][0];
#pragma unroll
            for (int ks = 0; ks < KS_POL; ks++) {
                if (ks < KS) {
                    const int j = ks * 16 + 2 * q;
                    const uint32_t bh0 = *reinterpret_cast<const uint32_t*>(rh + j), bh1 = *reinterpret_cast<const uint32_t*>(rh + j + 8);
                    const uint32_t bl0 = *reinterpret_cast<const uint32_t*>(rl + j), bl1 = *reinterpret_cast<const uint32_t*>(rl + j + 8);
                    mma_bf16_16816(c, ah[ks][0], ah[ks][1], ah[ks][2], ah[ks][3], bh0, bh1);
                    mma_bf16_16816(c, ah[ks][0], ah[ks][1], ah[ks][2], ah[ks][3], bl0, bl1);
                    mma_bf16_16816(c, al[ks][0], al[ks][1], al[ks][2], al[ks][3], bh0, bh1);
                }
            }
            const int pc = nt * 8 + 2 * q;                               // this lane's two positions (accumulator columns)
            if (pol) {
                if (pc < cnt) {
                    if (u0 < NPOL) logits[(base + pc) * NPOL + u0] = c[0];
                    if (u1 < NPOL) logits[(base + pc) * NPOL + u1] = c[2];
                }
                if (pc + 1 < cnt) {
                    if (u0 < NPOL) logits[(base + pc + 1) * NPOL + u0] = c[1];
                    if (u1 < NPOL) logits[(base + pc + 1) * NPOL + u1] = c[3];
                }
            } else {
                // value_fc2 on relu(hidden) (model.py:353-355): this lane's two units, then the eight unit rows of the tile
                float s0 = fmaf(fmaxf(c[2], 0.0f), w2b, fmaxf(c[0], 0.0f) * w2a), s1 = fmaf(fmaxf(c[3], 0.0f), w2b, fmaxf(c[1], 0.0f) * w2a);
#pragma unroll
                for (int o = 4; o < 32; o <<= 1) {
                    s0 += __shfl_xor_sync(0xFFFFFFFFu, s0, o);
                    s1 += __shfl_xor_sync(0xFFFFFFFFu, s1, o);
                }
                if (g == 0) { s_part[m][pc] = s0; s_part[m][pc + 1] = s1; }
            }
        }
    }
    __syncthreads();
    if (t < cnt) {
        float sum = P.b_v2;
#pragma unroll
        for (int m = 0; m < MT_VAL; m++) sum += s_part[m][t];
        value[base + t] = tanhf(sum);                                    // model.py:355
    }
}

}  // namespace hz

extern "C" int hz_net_heads_fc_active(const float* head_conv, const void* glob, int64_t n, const int32_t* n_active, int H,
                                      const float* w_pol_t, const float* b_pol, const float* w_v1_t, const float* b_v1,
                                      const float* w_v2, float b_v2, float* logits, float* value, void* stream) {
    if (n == 0) return HZ_OK;
    if ((uintptr_t)n_active & 3) return HZ_ERR_ARG;
    if (!head_conv || !glob || !w_pol_t || !b_pol || !w_v1_t || !b_v1 || !w_v2 || !logits || !value || n < 0) return HZ_ERR_ARG;
    if (H != hz::FH || (((uintptr_t)w_v1_t | (uintptr_t)w_pol_t) & 15)) return HZ_ERR_ARG;
    hz::HeadParams P{nullptr, nullptr, w_pol_t, b_pol, w_v1_t, b_v1, w_v2, b_v2, hz::FC, H};
    hz::k_heads_fc_mma<<<(unsigned)((n + hz::MB - 1) / hz::MB), hz::MTPB, 0, (cudaStream_t)stream>>>(
        head_conv, (const __nv_bfloat16*)glob, n, P, logits, value, n_active);
    return hz_launched(1);
}

extern "C" int hz_net_heads(const void* x, const void* glob, int64_t n, int C, int H, const float* w_conv,
                            const float* b_conv, const float* w_pol_t, const float* b_pol, const float* w_v1_t,
                            const float* b_v1, const float* w_v2, float b_v2, float* logits, float* value,
                            void* stream) {
    if (n == 0) return HZ_OK;
    if (!x || !glob || !w_conv || !b_conv || !w_pol_t || !b_pol || !w_v1_t || !b_v1 || !w_v2 || !logits || !value)
        return HZ_ERR_ARG;
    if (n < 0 || C <= 0 || (C % 8) != 0 || H <= 0 || (H % 2) != 0 || ((uintptr_t)x & 15)) return HZ_ERR_ARG;
    hz::HeadParams P{w_conv, b_conv, w_pol_t, b_pol, w_v1_t, b_v1, w_v2, b_v2, C, H};
    if (C == hz::FC && H == hz::FH && (((uintptr_t)w_v1_t | (uintptr_t)w_pol_t) & 15) == 0) {
        static bool attr_set[64] = {};   // the opt-in shared-memory size is per function and per device
        int dev = 0;
        cudaGetDevice(&dev);
        if (dev < 0 || dev >= 64 || !attr_set[dev]) {
            cudaError_t e = cudaFuncSetAttribute(hz::k_heads_p, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hz::FSMEM);
            if (e != cudaSuccess) return hz_record_launch(0, e);
            if (dev >= 0 && dev < 64) attr_set[dev] = true;
        }
        int64_t fgroups = (n + hz::FG - 1) / hz::FG;
        int fgrid = (int)(fgroups < 148 ? fgroups : 148);
        hz::k_heads_p<<<fgrid, hz::FTPB, hz::FSMEM, (cudaStream_t)stream>>>((const __nv_bfloat16*)x, (const __nv_bfloat16*)glob,
                                                                            n, P, logits, value);
        return hz_launched(1);
    }
    size_t smem = sizeof(float) * (size_t)(3 * C + hz::HP * hz::PIN + hz::HP * 80 + hz::HP * 8);
    int64_t groups = (n + hz::HP - 1) / hz::HP;
    int grid = (int)(groups < 148 * 4 ? groups : 148 * 4);
    hz::k_heads<<<grid, hz::HTPB, smem, (cudaStream_t)stream>>>((const __nv_bfloat16*)x, (const __nv_bfloat16*)glob, n, P,
                                                                logits, value);
    return hz_launched(1);
}
