// probe_core.cu — test-only launchers that run the bit-sliced primitives of csrc/hz_core.cuh directly, over whole
// input domains, next to plain references (tests/test_gpu_core_domain.py builds and loads this file).
//
// Every checking launcher counts the inputs where primitive and reference disagree in out[0] and stores the first
// 16 of them as records of 32 words at out[32 * (1 + slot)]; word 0 of a record says which comparison failed.  The
// references are naive loops over the host specification: packed.draw_pile for the draws, the oracle's legal set
// walked in ascending action order for a placement, eight single steps for a round.  The ref_* launchers run a
// reference alone, so that the test can check it against that specification too.
#include "../harmonies_alphazero_b200/csrc/hz_core.cuh"

using namespace hz;

namespace {

constexpr int REC_WORDS = 32, N_RECS = 16;

__device__ void report(uint32_t* out, const uint32_t* v, int nv) {
    const uint32_t slot = atomicAdd(out, 1u);
    if (slot >= N_RECS) return;
    for (int i = 0; i < nv && i < REC_WORDS; i++) out[REC_WORDS * (1 + slot) + i] = v[i];
}

// ---- nth_set_bit ---------------------------------------------------------------------------------------------------
__device__ int ref_nth(uint32_t m, int k) {
    for (int i = 0; i < 32; i++)
        if ((m >> i) & 1u) {
            if (k == 0) return i;
            k--;
        }
    return -1;
}

__global__ void k_nth_sweep(uint32_t* out) {
    const uint32_t m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= (1u << 23)) return;
    const int n = __popc(m);
    for (int k = 0; k < n; k++) {
        const int got = nth_set_bit(m, k), want = ref_nth(m, k);
        if (got != want) {
            const uint32_t v[5] = {1u, m, (uint32_t)k, (uint32_t)got, (uint32_t)want};
            report(out, v, 5);
        }
    }
}

__global__ void k_ref_nth(const uint32_t* m, const int32_t* k, int64_t n, int32_t* pos) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) pos[i] = ref_nth(m[i], k[i]);
}

// ---- draws: packed.draw_pile, tile by tile ---------------------------------------------------------------------
__device__ uint32_t ref_draw_pile(uint64_t& bag, uint64_t z) {
    int cnt[6];
    for (int t = 0; t < 6; t++) cnt[t] = (int)((bag >> (8 * t)) & 0xFFu);
    uint32_t code = 0;
    for (int j = 0; j < 3; j++) {
        int total = 0;
        for (int t = 0; t < 6; t++) total += cnt[t];
        if (total == 0) break;
        const uint64_t x = (z >> (21 * j)) & 0x1FFFFFu;
        int64_t r = (int64_t)((x * (uint64_t)total) >> 21);
        int t = 0;
        for (; t < 6; t++) {
            if (r < cnt[t]) break;
            r -= cnt[t];
        }
        cnt[t]--;
        code += 1u << (2 * t);
    }
    bag = 0;
    for (int t = 0; t < 6; t++) bag |= (uint64_t)cnt[t] << (8 * t);
    return code;
}

// bag_total, draw_pile and (where its range holds, 3 <= total <= 127) draw_pile3 against the reference
__device__ void check_draw(uint64_t bag, uint64_t z, uint32_t* out) {
    int ref_total = 0;
    for (int t = 0; t < 6; t++) ref_total += (int)((bag >> (8 * t)) & 0xFFu);
    uint64_t want_bag = bag;
    const uint32_t want = ref_draw_pile(want_bag, z);
    uint64_t got_bag = bag;
    uint32_t got = draw_pile(got_bag, z);
    const int total = bag_total(bag);
    uint32_t kind = total != ref_total ? 1u : (got != want || got_bag != want_bag) ? 2u : 0u;
    if (kind == 0 && total >= 3 && total <= 127) {
        uint32_t lo = (uint32_t)bag, hi = (uint32_t)(bag >> 32);
        got = draw_pile3(lo, hi, (uint32_t)total, z);
        got_bag = (uint64_t)lo | ((uint64_t)hi << 32);
        if (got != want || got_bag != want_bag) kind = 3u;
    }
    if (kind) {
        const uint32_t v[11] = {kind, (uint32_t)bag, (uint32_t)(bag >> 32), (uint32_t)z, (uint32_t)(z >> 32), got, want,
                                (uint32_t)got_bag, (uint32_t)(got_bag >> 32), (uint32_t)want_bag, (uint32_t)(want_bag >> 32)};
        report(out, v, 11);
    }
}

// every bag of 0..23, 0..19, 0..21, 0..23, 0..15, 0..19 tiles (the compositions within the initial bag), nz draws each
__global__ void k_draw_sweep(uint64_t seed, int nz, uint32_t* out) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int RADIX[6] = {24, 20, 22, 24, 16, 20};
    int64_t rem = idx;
    uint64_t bag = 0;
    for (int t = 0; t < 6; t++) {
        bag |= (uint64_t)(rem % RADIX[t]) << (8 * t);
        rem /= RADIX[t];
    }
    if (rem != 0) return;
    for (int i = 0; i < nz; i++) check_draw(bag, rand64(seed, (uint64_t)idx * (uint64_t)nz + (uint64_t)i), out);
}

__global__ void k_draw_list(const uint64_t* bags, const uint64_t* zs, int64_t n, uint32_t* out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) check_draw(bags[i], zs[i], out);
}

__global__ void k_ref_draw(const uint64_t* bags, const uint64_t* zs, int64_t n, uint32_t* codes, uint64_t* bags_out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t b = bags[i];
    codes[i] = ref_draw_pile(b, zs[i]);
    bags_out[i] = b;
}

// ---- place_random ------------------------------------------------------------------------------------------------
// The k-th legal placement (k = the policy draw's share of n, as the oracle's random_action takes it) from per-type
// legal masks, walked in ascending action order (type-major, then hex), put on the planes at the stack's height.
// Returns the hex's bit (0 when nothing is legal: planes and hand untouched).
__device__ uint32_t ref_place(uint32_t* b, uint32_t& hand, uint32_t rh, const uint32_t* masks) {
    int n = 0;
    for (int t = 0; t < 6; t++)
        if ((hand >> (2 * t)) & 3u)
            for (int h = 0; h < 23; h++) n += (masks[t] >> h) & 1u;
    if (n == 0) return 0;
    int k = (int)(((uint64_t)rh * (uint64_t)n) >> 32);
    for (int t = 0; t < 6; t++) {
        if (!((hand >> (2 * t)) & 3u)) continue;
        for (int h = 0; h < 23; h++) {
            if (!((masks[t] >> h) & 1u)) continue;
            if (k-- > 0) continue;
            int level = 0;
            while (level < 3 && (((b[3 * level] | b[3 * level + 1] | b[3 * level + 2]) >> h) & 1u)) level++;
            for (int q = 0; q < 3; q++)
                if (((uint32_t)(t + 1) >> q) & 1u) b[3 * level + q] |= 1u << h;
            hand -= 1u << (2 * t);
            return 1u << h;
        }
    }
    return 0;
}

__device__ void check_place(const uint32_t* board, const uint32_t* masks, uint32_t hand0, uint32_t rh, uint32_t kind_k,
                            uint32_t board_id, uint32_t* out) {
    uint32_t gb[9], wb[9], gh = hand0, wh = hand0;
    for (int q = 0; q < 9; q++) gb[q] = wb[q] = board[q];
    const uint32_t got = place_random(gb, gh, rh), want = ref_place(wb, wh, rh, masks);
    int bad = got != want || gh != wh ? 9 : -1;
    for (int q = 0; q < 9 && bad < 0; q++)
        if (gb[q] != wb[q]) bad = q;
    if (bad >= 0) {
        const uint32_t v[10] = {kind_k, board_id, hand0, rh, got, want, gh, wh, (uint32_t)bad, bad < 9 ? gb[bad] ^ wb[bad] : 0u};
        report(out, v, 10);
    }
}

// one thread per (board, hand code 0..4095): both edge values of the policy draw for every k < n, the two extreme
// draws when n == 0.  evals counts the placements compared.
__global__ void k_place_sweep(const uint32_t* boards, const uint32_t* masks, int nb, uint32_t* out, unsigned long long* evals) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)nb * 4096) return;
    const int bi = (int)(idx >> 12);
    const uint32_t hand = (uint32_t)idx & 4095u;
    const uint32_t* b = boards + 9 * bi;
    const uint32_t* m = masks + 6 * bi;
    uint32_t n = 0;
    for (int t = 0; t < 6; t++)
        if ((hand >> (2 * t)) & 3u) n += __popc(m[t]);
    unsigned long long count = 0;
    if (n == 0) {
        check_place(b, m, hand, 0u, 0u, (uint32_t)bi, out);
        check_place(b, m, hand, 0xFFFFFFFFu, 0u, (uint32_t)bi, out);
        count = 2;
    }
    for (uint32_t k = 0; k < n; k++) {
        // the smallest and the largest rh with floor(rh * n / 2^32) == k
        const uint64_t lo = (((uint64_t)k << 32) + n - 1) / n, hi = ((((uint64_t)k + 1) << 32) + n - 1) / n - 1;
        check_place(b, m, hand, (uint32_t)lo, 1u + k, (uint32_t)bi, out);
        check_place(b, m, hand, (uint32_t)hi, 1u + k, (uint32_t)bi, out);
        count += 2;
    }
    atomicAdd(evals, count);
}

__global__ void k_ref_place(const uint32_t* boards, const uint32_t* masks, const uint32_t* hands, const uint32_t* rhs,
                            int64_t n, uint32_t* res) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t b[9], hand = hands[i];
    for (int q = 0; q < 9; q++) b[q] = boards[9 * i + q];
    const uint32_t bit = ref_place(b, hand, rhs[i], masks + 6 * i);
    for (int q = 0; q < 9; q++) res[11 * i + q] = b[q];
    res[11 * i + 9] = hand;
    res[11 * i + 10] = bit;
}

// ---- playout_round against eight playout_step<P, true> ------------------------------------------------------------
// flags[i]: bit 0 round_ready, bit 1 playout_round returned true
constexpr int RTPB_PROBE = 64;
__global__ void __launch_bounds__(RTPB_PROBE) k_round(const uint32_t* recs, int64_t n, uint32_t* out, uint32_t* flags) {
    __shared__ NbrLut lut;
    __shared__ __align__(16) uint64_t rtab_s[RTAB_N];
    build_nbr_lut(&lut);
    build_rand_table(rtab_s);
    const RandTab rtab = rand_table_handle(rtab_s);
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * RTPB_PROBE + threadIdx.x;
    if (i >= n) return;
    State s0;
    for (int q = 0; q < SW; q++) s0.w[q] = recs[32 * i + q];
    const bool ready = round_ready(s0);
    bool ok = false;
    if (ready) {
        State a = s0, b = s0;
        ok = playout_round(a, rtab);
        uint32_t kind = 0;
        if (ok) {
            for (int j = 0; j < 8 && kind == 0; j++) {
                const bool st = player_of(b) ? playout_step<1, true>(b, &lut, rtab) : playout_step<0, true>(b, &lut, rtab);
                if (!st) kind = 1;   // a step found no legal move inside a round the straight line took
            }
        } else {
            b = s0;                  // false: the record must be untouched
        }
        int word = -1;
        for (int q = 0; q < SW && word < 0; q++)
            if (a.w[q] != b.w[q]) word = q;
        if (kind == 0 && word >= 0) kind = ok ? 2u : 3u;
        if (kind) {
            const uint32_t v[6] = {kind, (uint32_t)i, (uint32_t)word, word >= 0 ? a.w[word] : 0u, word >= 0 ? b.w[word] : 0u,
                                   ok ? 1u : 0u};
            report(out, v, 6);
        }
    }
    flags[i] = (ready ? 1u : 0u) | (ok ? 2u : 0u);
}

inline unsigned blocks(int64_t n, int tpb) { return (unsigned)((n + tpb - 1) / tpb); }

}  // namespace

// ---- C ABI: device pointers in, cudaError_t out (after a device synchronise) ----------------------------------------
extern "C" {
int probe_nth_sweep(uint32_t* out) {
    k_nth_sweep<<<(1u << 23) / 256, 256>>>(out);
    return (int)cudaDeviceSynchronize();
}
int probe_ref_nth(const uint32_t* m, const int32_t* k, int64_t n, int32_t* pos) {
    k_ref_nth<<<blocks(n, 256), 256>>>(m, k, n, pos);
    return (int)cudaDeviceSynchronize();
}
int probe_draw_sweep(uint64_t seed, int nz, uint32_t* out) {
    const int64_t n = 24ll * 20 * 22 * 24 * 16 * 20;
    k_draw_sweep<<<blocks(n, 256), 256>>>(seed, nz, out);
    return (int)cudaDeviceSynchronize();
}
int probe_draw_list(const uint64_t* bags, const uint64_t* zs, int64_t n, uint32_t* out) {
    k_draw_list<<<blocks(n, 256), 256>>>(bags, zs, n, out);
    return (int)cudaDeviceSynchronize();
}
int probe_ref_draw(const uint64_t* bags, const uint64_t* zs, int64_t n, uint32_t* codes, uint64_t* bags_out) {
    k_ref_draw<<<blocks(n, 256), 256>>>(bags, zs, n, codes, bags_out);
    return (int)cudaDeviceSynchronize();
}
int probe_place_sweep(const uint32_t* boards, const uint32_t* masks, int nb, uint32_t* out, unsigned long long* evals) {
    k_place_sweep<<<blocks((int64_t)nb * 4096, 128), 128>>>(boards, masks, nb, out, evals);
    return (int)cudaDeviceSynchronize();
}
int probe_ref_place(const uint32_t* boards, const uint32_t* masks, const uint32_t* hands, const uint32_t* rhs, int64_t n,
                    uint32_t* res) {
    k_ref_place<<<blocks(n, 256), 256>>>(boards, masks, hands, rhs, n, res);
    return (int)cudaDeviceSynchronize();
}
int probe_round(const uint32_t* recs, int64_t n, uint32_t* out, uint32_t* flags) {
    k_round<<<blocks(n, RTPB_PROBE), RTPB_PROBE>>>(recs, n, out, flags);
    return (int)cudaDeviceSynchronize();
}
}
