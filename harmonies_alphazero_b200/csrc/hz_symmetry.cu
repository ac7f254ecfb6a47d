// hz_symmetry.cu — the game's symmetry group on batches (sm_100a): hz_sym_states transforms packed records,
// hz_sym_actions permutes [n,143] policy / visit / mask rows (include/harmonies_b200.h "Game symmetries").
//
// Both are bandwidth kernels.  hz_sym_states is one thread per record: the 18 plane words are rebuilt bit by bit from
// the inverse hex map (23 x 18 bit moves in registers, the map of the record's board part read from shared memory),
// which costs fewer instructions per record than the warp-per-record ballot form the search uses on its staged leaf
// (hz_sym.cuh: warp_sym_word, 18 shuffles + 18 ballots per record).  hz_sym_actions writes each output element once,
// out[i][a'] = x[i][sigma^-1(a')], a gather inside the row, so the stores are coalesced.
#include "hz_common.cuh"
#include "hz_sym.cuh"

namespace hz {

constexpr int STPB = 128;

__global__ void __launch_bounds__(STPB) k_sym_states(const uint4* in, int64_t n, const uint16_t* sym, uint4* out) {
    __shared__ uint8_t inv[4][24];
    if (threadIdx.x < 4 * 23) inv[threadIdx.x / 23][threadIdx.x % 23] = SYM_HEX_INV_G[threadIdx.x / 23][threadIdx.x % 23];
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * STPB + threadIdx.x;
    if (i >= n) return;
    uint32_t w[32];
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const uint4 v = in[i * 8 + k];
        w[4 * k] = v.x; w[4 * k + 1] = v.y; w[4 * k + 2] = v.z; w[4 * k + 3] = v.w;
    }
    const int g = sym[i], b = g & 3;
    if (b != 0) {
        uint32_t o[18];
#pragma unroll
        for (int k = 0; k < 18; k++) o[k] = 0;
#pragma unroll
        for (int h = 0; h < HZ_NUM_HEXES; h++) {
            const uint32_t s = inv[b][h];
#pragma unroll
            for (int k = 0; k < 18; k++) o[k] |= ((w[k] >> s) & 1u) << h;
        }
#pragma unroll
        for (int k = 0; k < 18; k++) w[k] = o[k];
    }
    if (g >> 2) sym_pile_words(w[HZ_W_PILES01], w[HZ_W_PILES23], w[HZ_W_PILE4H], w[HZ_W_BAG1META], g);
#pragma unroll
    for (int k = 0; k < 8; k++) out[i * 8 + k] = make_uint4(w[4 * k], w[4 * k + 1], w[4 * k + 2], w[4 * k + 3]);
}

// E = element type (uint32_t for fp32 / int32, uint16_t for int16): out[i][a'] = x[i][src(a')].  A block takes AROWS rows:
// their element (board part, n_piles, pile permutation) and the hex map are staged in shared memory once, and the
// block's threads then walk the rows' 143 * AROWS contiguous outputs with 32-bit in-block indices (the divisions by the
// constants 143 and 23 become multiplies), so the stores are coalesced and the gathered loads stay inside the block's rows.
constexpr int ATPB = 256, AROWS = 16;
template <typename E>
__global__ void __launch_bounds__(ATPB) k_sym_actions(const E* x, int64_t n, const uint16_t* sym, const uint4* states, int inverse,
                                                       E* out) {
    __shared__ uint8_t hex[4][24];
    __shared__ uint32_t rinfo[AROWS];                  // board part | n_piles << 2 | packed pile permutation << 8
    const int64_t row0 = (int64_t)blockIdx.x * AROWS;
    const int rows = (int)(n - row0 < AROWS ? n - row0 : AROWS);
    // forward: out[sigma(a)] = x[a], so out[a'] = x[sigma^-1(a')] (inverse tables); inverse: out[a'] = x[sigma(a')]
    if (threadIdx.x < 4 * 23) {
        const int b = threadIdx.x / 23, h = threadIdx.x % 23;
        hex[b][h] = inverse ? SYM_HEX_G[b][h] : SYM_HEX_INV_G[b][h];
    }
    if (threadIdx.x < rows) {
        const int64_t row = row0 + threadIdx.x;
        const int g = sym[row];
        int m = (int)((reinterpret_cast<const uint32_t*>(states + row * 8)[HZ_W_BAG1META] >> 16) & 0xFFu);
        m = m < 5 ? m : 5;
        rinfo[threadIdx.x] = (uint32_t)(g & 3) | ((uint32_t)m << 2) | (sym_pile_perm(g, m, inverse == 0) << 8);
    }
    __syncthreads();
    const E* xb = x + row0 * HZ_ACTION_SIZE;
    E* ob = out + row0 * HZ_ACTION_SIZE;
    const uint32_t total = (uint32_t)rows * HZ_ACTION_SIZE;
    for (uint32_t e = threadIdx.x; e < total; e += ATPB) {
        const uint32_t r = e / HZ_ACTION_SIZE, a = e - r * HZ_ACTION_SIZE;
        const uint32_t info = rinfo[r];
        uint32_t src;
        if (a < 5) {
            src = a < ((info >> 2) & 7u) ? (info >> (8 + 3 * a)) & 7u : a;
        } else {
            const uint32_t t = (a - 5) / 23, h = a - 5 - 23 * t;
            src = 5 + 23 * t + hex[info & 3u][h];
        }
        ob[e] = xb[r * HZ_ACTION_SIZE + src];
    }
}

}  // namespace hz

using namespace hz;

static inline int sym_blocks(int64_t n) { return (int)((n + STPB - 1) / STPB); }

extern "C" {

int hz_sym_states(const void* states, int64_t n, const uint16_t* sym, void* out, void* stream) {
    if (n == 0) return HZ_OK;
    if (!states || !sym || !out || n < 0) return HZ_ERR_ARG;
    k_sym_states<<<sym_blocks(n), STPB, 0, (cudaStream_t)stream>>>((const uint4*)states, n, sym, (uint4*)out);
    return hz_launched(1);
}

int hz_sym_actions(const void* x, int64_t n, int dtype, const uint16_t* sym, const void* states, int inverse, void* out,
                   void* stream) {
    if (dtype != HZ_DTYPE_F32 && dtype != HZ_DTYPE_I32 && dtype != HZ_DTYPE_I16) return HZ_ERR_ARG;
    if (n == 0) return HZ_OK;
    if (!x || !sym || !states || !out || n < 0 || x == out) return HZ_ERR_ARG;
    const int blocks = (int)((n + AROWS - 1) / AROWS);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == HZ_DTYPE_F32 || dtype == HZ_DTYPE_I32)
        k_sym_actions<uint32_t><<<blocks, ATPB, 0, st>>>((const uint32_t*)x, n, sym, (const uint4*)states, inverse,
                                                                    (uint32_t*)out);
    else
        k_sym_actions<uint16_t><<<blocks, ATPB, 0, st>>>((const uint16_t*)x, n, sym, (const uint4*)states, inverse,
                                                                    (uint16_t*)out);
    return hz_launched(1);
}

}  // extern "C"
