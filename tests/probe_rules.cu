// probe_rules.cu — test-only launchers for the engine's closed-form rules in csrc/hz_core.cuh that the public entry
// points reach only through other code (tests/test_gpu_rules_domain.py builds and loads this file):
//
//   - the neighbour expansion (nbr_alu, the shared-memory LUT) and the six direction pulls on every 23-bit mask, next to
//     loops over neighbour tables that the test derives from the axial coordinates;
//   - score_board with both ways of scoring a water component of >= 5 hexes: in place (NoWaterQueue) and through a block
//     queue that cannot overflow plus resolve_water.  hz_score mixes the two by how full a block's queue gets.
//
// A checking launcher counts the masks where primitive and reference disagree in out[0] and stores the first 16 of them
// as records of 32 words at out[32 * (1 + slot)]; word 0 of a record says which comparison failed.
#include "../harmonies_alphazero_b200/csrc/hz_core.cuh"

using namespace hz;

namespace {

constexpr int REC_WORDS = 32, N_RECS = 16;

__device__ void report(uint32_t* out, const uint32_t* v, int nv) {
    const uint32_t slot = atomicAdd(out, 1u);
    if (slot >= N_RECS) return;
    for (int i = 0; i < nv && i < REC_WORDS; i++) out[REC_WORDS * (1 + slot) + i] = v[i];
}

// ---- neighbour expansion and direction pulls -------------------------------------------------------------------------
// nbr_masks[i]: the hexes adjacent to hex i; dir_nb[6 * 23]: per direction E, W, S, N, NE, SW (constants.AXIAL_DIRECTIONS
// order), hex i's neighbour in that direction or -1.  kind 1..2: nbr_alu / LUT against the union of nbr_masks; 3..8: the
// pull of direction kind - 3 against its table.
__global__ void k_nbr_sweep(const uint32_t* nbr_masks, const int32_t* dir_nb, uint32_t* out) {
    __shared__ NbrLut lut;
    __shared__ uint32_t snb[23];
    __shared__ int32_t sdir[6 * 23];
    build_nbr_lut(&lut);
    for (int e = threadIdx.x; e < 23; e += blockDim.x) snb[e] = nbr_masks[e];
    for (int e = threadIdx.x; e < 6 * 23; e += blockDim.x) sdir[e] = dir_nb[e];
    __syncthreads();
    const uint32_t m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= (1u << 23)) return;
    uint32_t want = 0;
    for (int i = 0; i < 23; i++)
        if ((m >> i) & 1u) want |= snb[i];
    uint32_t got[8] = {nbr_alu(m), nbr(&lut, m), pull_E(m), pull_W(m), pull_S(m), pull_N(m), pull_NE(m), pull_SW(m)};
    uint32_t ref[8] = {want, want, 0, 0, 0, 0, 0, 0};
    for (int d = 0; d < 6; d++)
        for (int i = 0; i < 23; i++) {
            const int j = sdir[d * 23 + i];
            if (j >= 0 && ((m >> j) & 1u)) ref[2 + d] |= 1u << i;
        }
    for (int k = 0; k < 8; k++)
        if (got[k] != ref[k]) {
            const uint32_t v[4] = {1u + (uint32_t)k, m, got[k], ref[k]};
            report(out, v, 4);
        }
}

// ---- score_board with and without the water queue ---------------------------------------------------------------------
// k_score's layout (one thread per record, both boards), with a queue of 8 entries per thread: a board has at most four
// water components of >= 5 hexes, so no push can fail.  pushes[block] = the block's queue count.
constexpr int STPB = 128;
template <bool QUEUE>
__global__ void __launch_bounds__(STPB) k_score_probe(const uint32_t* states, int64_t n, int16_t* terms, int32_t* pushes) {
    __shared__ NbrLut lut;
    __shared__ WaterQueue<8 * STPB, 2 * STPB> wq;
    build_nbr_lut(&lut);
    water_queue_init(&wq);
    __syncthreads();
    const int64_t g = (int64_t)blockIdx.x * STPB + threadIdx.x;
    int t[2][5];
    if (g < n) {
        for (int pl = 0; pl < 2; pl++) {
            Board b;
            for (int k = 0; k < 9; k++) b.p[k] = states[g * 32 + pl * 9 + k];
            if (QUEUE) score_board(&lut, b, t[pl], &wq, (int)threadIdx.x * 2 + pl);
            else score_board(&lut, b, t[pl]);
        }
    }
    __syncthreads();
    if (QUEUE) resolve_water(&lut, &wq);
    __syncthreads();
    if (threadIdx.x == 0) pushes[blockIdx.x] = wq.count;
    if (g >= n) return;
    for (int pl = 0; pl < 2; pl++) {
        t[pl][4] += wq.extra[threadIdx.x * 2 + pl];
        for (int k = 0; k < 5; k++) terms[(g * 2 + pl) * 5 + k] = (int16_t)t[pl][k];
    }
}

inline unsigned blocks(int64_t n, int tpb) { return (unsigned)((n + tpb - 1) / tpb); }

}  // namespace

// ---- C ABI: device pointers in, cudaError_t out (after a device synchronise) ----------------------------------------
extern "C" {
int probe_nbr_sweep(const uint32_t* nbr_masks, const int32_t* dir_nb, uint32_t* out) {
    k_nbr_sweep<<<(1u << 23) / 256, 256>>>(nbr_masks, dir_nb, out);
    return (int)cudaDeviceSynchronize();
}
// queue 0: every large water component scored in place; 1: every one through the queue and resolve_water
int probe_score(const uint32_t* states, int64_t n, int queue, int16_t* terms, int32_t* pushes) {
    if (queue) k_score_probe<true><<<blocks(n, STPB), STPB>>>(states, n, terms, pushes);
    else k_score_probe<false><<<blocks(n, STPB), STPB>>>(states, n, terms, pushes);
    return (int)cudaDeviceSynchronize();
}
}
