// hz_tower.cu — hand-written sm_100a 3x3 convolution for the residual tower of the reference
// network (model.py:325-357 stem conv+bn+relu, ResidualBlock.forward model.py:380-392), BatchNorm
// folded, bf16 operands, fp32 accumulation in tensor memory.  SURVEY.md §8 row f4.
//
// Formulation (per layer):  out[o][p] = sum over taps t=(dy,dx), channels i of W_t[o][i] * in[i][p + s(t)]
//   * tcgen05.mma, M = 128 output channels (A = one tap's weight tile, K-major SWIZZLE_128B),
//     N = board positions (B = a window of the activation tile, K-major SWIZZLE_128B), accumulators
//     in TMEM: lane = output channel, column = position.
//   * activations live in HBM as 16-board tiles in exactly the byte image the tensor core reads
//     from shared memory, so one bulk copy (TMA, cp.async.bulk) brings a tile half in.  Positions
//     are cell-major: p = cell*16 + board.  Two images exist:
//       T16  (every layer's output, the residual convolutions' input): MN-major, no swizzle —
//            8-channel group kg at kg*8960 bytes, inside it 8-position group pg at pg*128, inside
//            that a core matrix [8 channels][8 positions] with positions contiguous.  An epilogue
//            thread owns one output channel and therefore writes 16 boards of a cell as two
//            16-byte vectors (and reads the residual the same way).
//       T16K (the stem's input, written by the leaf encoder 8 channels = 16 bytes at a time):
//            K-major SWIZZLE_128B, row p of 128 bytes = 64 channels, group g at g ^ (p & 7).
//     With cells outermost a tap is a shift by whole cells: the B operand of tap (dy,dx) for
//     output board-row r is the SAME resident tile read through a descriptor whose start address
//     moved by ((r+dy)*7 + max(dx,0)) cells.
//   * taps that fall off the 5x7 board are never multiplied: rows with r+dy outside 0..4 skip the
//     tap, and a dx = -1 / +1 tap covers only the six cells x = 1..6 / 0..5 (N = 96 instead of 112,
//     accumulator window moved by 16 columns).  Executed MACs = 247/315 of a zero-padded conv.
//   * a whole tile stays in shared memory for all nine taps (one HBM/L2 read per layer); the
//     weights stream through a 5-stage ring (16 KB = one tap x one channel half per stage).
//   * TMEM holds 512 positions (4 board rows of 16 boards) but a tile has 560, so a tile is two
//     passes over the weight stream: board rows {0,1,2} then {3,4}.  Row accumulators live in four
//     128-column units: rows 0..3 own units 0..3 and row 4 shares unit 0 with row 0.  The tap order
//     makes that free of stalls: pass 0 runs dy = +1, 0, -1, so row 0 (which has no dy = -1 tap) is
//     complete and drained before pass 1 starts; pass 1 runs dy = -1, 0, +1, so row 4 (no dy = +1)
//     is drained before the next tile's row 0 needs the unit.  The epilogue of one row therefore
//     always overlaps the MMAs of the others.
//   * hz_tower_forward_heads: clusters of two CTAs take pairs of neighbouring tiles of one layer and share the weight
//     stream: each CTA loads half of every stage and multicasts it to both (cluster mode, see Params::pair).
//   * warp roles: 0 = weight producer, 1 and 12 = MMA issuers (alternating weight stages), 2 =
//     activation producer, 3 = TMEM allocator + work scheduler, 4..11 = epilogue (bias + residual +
//     ReLU + bf16, thread = output channel).
#include "hz_common.cuh"
#include "hz_sm100.cuh"

namespace hz {
namespace tower {
using namespace hz::sm100;

constexpr int G = 16;                          // boards per tile
constexpr int CELLS = 35, BROWS = 5, BCOLS = 7;
constexpr int TILE_ROWS = CELLS * G;           // 560 rows of 128 bytes per channel half
constexpr int KH_BYTES = TILE_ROWS * 128;      // 71,680: one 64-channel half of a tile (either image)
constexpr int KG_BYTES = (TILE_ROWS / 8) * 128; // 8,960: one 8-channel group of a T16 tile (70 position groups)
constexpr int ROW_BYTES = BCOLS * G * 128;     // 14,336: one board row of one channel half
constexpr int W_BYTES = 128 * 128;             // 16,384: [128 out][64 in] bf16
constexpr int NSTAGE = 5;
constexpr int NUNIT = 4, UNIT_COLS = 128;
constexpr int NTHREADS = 416;                  // 4 control warps + 8 epilogue warps + the second MMA issuer
constexpr int OFF_X = 0;
constexpr int OFF_W = 2 * KH_BYTES;
constexpr int OFF_BAR = OFF_W + NSTAGE * W_BYTES;
constexpr int SMEM_BYTES = OFF_BAR + 512 + 1024;   // barriers + alignment slack

// barrier indices
constexpr int B_WFULL = 0, B_WEMPTY = NSTAGE, B_AFULL = 2 * NSTAGE, B_AEMPTY = 2 * NSTAGE + 2, B_TFULL = 2 * NSTAGE + 4,
              B_TEMPTY = 2 * NSTAGE + 4 + NUNIT, B_DONE = 2 * NSTAGE + 4 + 2 * NUNIT, B_QFULL = B_DONE + 1, B_QEMPTY = B_QFULL + 2,
              N_BARS = B_QEMPTY + 2;

// tap = ky*3 + kx (dy = ky-1, dx = kx-1).  Within a dy group the dx = 0 tap comes first: the first
// MMA into a row accumulator overwrites it and must cover all 112 columns.
//
// A tile's five board rows do not fit the four accumulator units at once, so a work item is a sequence of
// SEGMENTS, each a list of taps applied to a range of rows, run per channel half (segment-outer, half-inner):
// rows {0,1,2} + {3,4}, 9 taps each:
//   seg 0: rows 0..2, dy = +1, 0, -1  -> row 0 (no dy = -1 tap) completes after two thirds of the segment
//   seg 1: rows 3..4, dy = -1, 0, +1  -> row 4 (no dy = +1 tap) completes after two thirds of the segment
//   so the unit rows 0 and 4 share is always drained before its next tenant arrives.
// (A 4 + 1 split needs 30 weight stages per item instead of 36, but the single-row segment's stages are 4 MMAs (~210
// tensor cycles) against a weight ring that delivers one 16 KB stage per >= 400 cycles: measured 415-420 us against 394.)
constexpr int NSEG = 2;
__host__ __device__ constexpr int seg_nt(int) { return 9; }
__host__ __device__ constexpr int seg_r0(int seg) { return seg ? 3 : 0; }
__host__ __device__ constexpr int seg_r1(int seg) { return seg ? 5 : 3; }
__host__ __device__ constexpr int tap_at(int seg, int ti) {
    constexpr int O[2][9] = {{7, 6, 8, 4, 3, 5, 1, 0, 2}, {1, 0, 2, 4, 3, 5, 7, 6, 8}};
    return O[seg][ti];
}
__constant__ int8_t SEG_TAPS[2][9] = {{7, 6, 8, 4, 3, 5, 1, 0, 2}, {1, 0, 2, 4, 3, 5, 7, 6, 8}};
__constant__ int8_t EPI_ORDER[5] = {0, 1, 2, 4, 3};  // order in which the row accumulators complete
// does stage (seg, ti) multiply into board row r?  (rows of the segment whose source row r + dy is on the board)
__host__ __device__ constexpr bool touches(int seg, int ti, int r) {
    const int dy = tap_at(seg, ti) / 3 - 1;
    return r >= seg_r0(seg) && r < seg_r1(seg) && r + dy >= 0 && r + dy < BROWS;
}
// is (seg, ti) the first / the last stage of the item's sequence that touches row r?  (for one channel half; the first
// touch of the first half overwrites the accumulator, the last touch of the last half completes it)
__host__ __device__ constexpr bool first_touch(int seg, int ti, int r) {
    if (!touches(seg, ti, r)) return false;
    for (int s2 = 0; s2 <= seg; s2++)
        for (int t2 = 0; t2 < (s2 == seg ? ti : seg_nt(s2)); t2++)
            if (touches(s2, t2, r)) return false;
    return true;
}
__host__ __device__ constexpr bool last_touch(int seg, int ti, int r) {
    if (!touches(seg, ti, r)) return false;
    for (int s2 = seg; s2 < NSEG; s2++)
        for (int t2 = (s2 == seg ? ti + 1 : 0); t2 < seg_nt(s2); t2++)
            if (touches(s2, t2, r)) return false;
    return true;
}
// accumulator unit of board row r and how many times the unit has been used before (tile iteration it)
__device__ __forceinline__ int unit_of(int r) { return r == 4 ? 0 : r; }
__device__ __forceinline__ int use_of(int r, int it) { return r == 0 ? 2 * it : r == 4 ? 2 * it + 1 : it; }

constexpr int MAX_LAYERS = 20;   // stem + 8 residual blocks = 17
constexpr int N_CONSUMERS = 12;  // roles that read the work-item queue: weight producer, activation producer, 2 MMA warps, 8 epilogue warps
constexpr unsigned FLAG_DONE = 8; // a tile's layer output is complete when its 8 epilogue warps have signalled

struct Layer {
    const uint8_t* w;      // weight tiles [9][nkh][128][128 B]
    const float* bias;     // [128]
    int in_buf, res_buf, out_buf;   // indices into Params::buf; res_buf < 0: no residual
    int nkh, kmajor, relu; // input channel halves; input image T16K (stem) or T16
    // head != 0: the 1x1 head convolutions (model.py:340-343,349-351) as ONE tap: w = [nkh][128][128 B] with rows 0..2 the
    // bf16 high parts of the three head filters and rows 3..5 their low parts (w = hi + lo: fp32-weight accuracy), bias[3],
    // output relu(conv + bias) as fp32 into head_out[tile][filter 0..2][cell][board] (1,680 floats per tile)
    int head;
    float* head_out;
};
// One launch runs layers[0..n_layers) for all tiles.  Work item i = (layer i / n_tiles, tile i % n_tiles);
// boards are independent, so item (l, t) depends on item (l-1, t) only.  With `sched` the CTAs take items
// from a global READY QUEUE: it starts with the stem items, and the last of the 8 epilogue warps to finish
// item (l, t) appends (l+1, t).  An item is therefore handed out only when its input is complete (no
// dependency stalls, and its tile can be prefetched while the previous item is still in flight), and the
// load balances to within one item per CTA (a static tile-to-CTA map leaves 40 of 148 CTAs idle half the
// time at 256 tiles).  Every queue slot below n_items is filled exactly once, so a scheduler that drew
// slot s only ever waits for the s-th completion, which some running CTA is producing: no deadlock (all
// CTAs are co-resident: grid <= SM count, one CTA per SM).  Without `sched` (single layer): static map.
struct Params {
    uint8_t* buf[4];       // activation tile buffers (T16; a kmajor layer's input buffer is T16K with one half)
    Layer layers[MAX_LAYERS];
    int n_layers, n_tiles;
    unsigned int* sched;   // ready queue (see hz_tower_forward_heads): [0] head, [1] tail, [2 + item] completion count, [2 + n_items + slot] queue
    int dbg;               // profiling only (hz_tower_set_debug): 1 skip MMAs, 2 skip epilogue memory traffic, 4 skip weight copies, 8 skip activation copies
    unsigned int* fault;
    unsigned long long* trace;   // profiling only (hz_tower_set_trace): SM-clock timestamps of CTA 0's roles
    const int* n_active;         // device word (nullable): only the tiles that hold boards 0..*n_active-1 are computed
    // cluster mode (hz_tower_forward_heads, clusters of `pair` = 2 CTAs; 0 = off): a work item is a group of neighbouring tiles
    // of one layer, one tile per CTA, so all CTAs of the cluster stream the same weights: each loads its share of every weight
    // stage and multicasts it to all of them (the weights are 57 % of what a launch pulls through L2).  mailbox: [cluster][64]
    // words through which CTA 0 of a cluster tells the others which item it drew.
    int pair;
    unsigned int* mailbox;
};
// tiles to compute: all of them, or those of the active board prefix (every thread of the grid reads the same word)
__device__ __forceinline__ int tiles_of(const int* n_active, int n_tiles) {
    if (!n_active) return n_tiles;
    const int n = (*n_active + G - 1) / G;
    return n < 0 ? 0 : n < n_tiles ? n : n_tiles;
}
// trace slots (CTA 0 only, 4096 uint64): [0] start, [1] end (SM clock), [2] start, [3] end (globaltimer, ns);
// MMA warp per weight stage i < 600: [16+3i] before the wait on the stage, [+1] after it, [+2] after the MMAs
// and commits were issued; weight producer [2000+i] when it issues stage i; epilogue warp 4 per row j < 200:
// [2700+4j] before the accumulator wait, [+1] after, [+2] after the TMEM loads, [+3] after the stores;
// activation producer [3600+j] when it issues half j.
// compiled in with -DHZ_TOWER_TRACE=1 only (profiles/tower_trace.py): the time stamps cost instruction-cache space
#ifndef HZ_TOWER_TRACE
#define HZ_TOWER_TRACE 0
#endif
#if HZ_TOWER_TRACE
#define HZ_TRACE(slot)                                                                  \
    do {                                                                                \
        if (P.trace && blockIdx.x == 0 && lane == 0 && (slot) < 4096) P.trace[slot] = clock64(); \
    } while (0)
#define HZ_CTRACE(slot)                                                                 \
    do {                                                                                \
        if (c.trace && c.nstage < 600) c.trace[slot] = clock64();                       \
    } while (0)
#else
#define HZ_TRACE(slot) do { } while (0)
#define HZ_CTRACE(slot) do { } while (0)
#endif
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// B operand, MN-major without swizzle: core matrices of [8 channels][8 positions]; LBO = stride
// between 8-channel groups (K direction), SBO = stride between 8-position groups (N direction)
__device__ __forceinline__ uint64_t smem_desc_t16(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
    d |= (uint64_t)((KG_BYTES >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((128 >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}
// max(x, 0) and round-to-nearest-even to bf16 in one instruction (NaN -> canonical NaN, as cuDNN's ReLU epilogue)
__device__ __forceinline__ uint32_t pack_bf16x2_relu(float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}

// ---- MMA issue, fully unrolled -------------------------------------------------------------------
// One thread issues ~312 MMAs of ~50 tensor-core cycles each per tile, so the issue path has to be
// a handful of instructions per MMA: the whole warp runs the (warp-uniform) control flow, taps /
// rows / k-steps are compile-time, descriptors are a 32-bit add on a precomputed low word, and only
// the tcgen05 instructions themselves sit behind elect.sync.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
// descriptor words: hi is constant per operand kind, lo = encoded start address (+ LBO field)
constexpr uint32_t DESC_HI_SW128 = (1024u >> 4) | (1u << 14) | (2u << 29);   // SBO 1024, version 1, SWIZZLE_128B
constexpr uint32_t DESC_LO_SW128 = 1u << 16;                                  // LBO field (unused) = 1
constexpr uint32_t DESC_HI_T16 = (128u >> 4) | (1u << 14);                    // SBO 128, version 1, no swizzle
constexpr uint32_t DESC_LO_T16 = (uint32_t)(KG_BYTES >> 4) << 16;             // LBO = 8-channel group stride
__device__ __forceinline__ uint64_t desc64(uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; }

// the MMAs of one weight stage (tap, channel half): 4 k-steps x the rows of the pass the tap touches
template <bool KMAJOR, int PASS, int TI, int K0, int K1>
__device__ __forceinline__ void issue_stage(uint32_t a_lo, uint32_t b_lo, uint32_t tbase, uint32_t acc_first) {
    constexpr int tap = tap_at(PASS, TI), dy = tap / 3 - 1, dx = tap % 3 - 1;
    constexpr int r0 = seg_r0(PASS), r1 = seg_r1(PASS);
    constexpr uint32_t idesc = idesc_bf16_f32(128, dx ? 96 : 112) | (KMAJOR ? 0u : (1u << 16));
    // rows of the segment this tap touches: [ra, rb) (always a contiguous range)
    constexpr int ra = (r0 + dy < 0) ? -dy : r0, rb = (r1 - 1 + dy >= BROWS) ? BROWS - dy : r1;
    static_assert(ra < rb, "a stage without rows");
    // the k loop is NOT unrolled: with it unrolled the issue code of a residual layer is 41 KB, more than the instruction
    // cache keeps beside the epilogue, and every change of pass stalled both issuers on instruction fetch (role timeline,
    // profiles/tower_trace.py: 2-14 thousand cycles at the first stage of pass 1 of every work item; tower 435 -> 400 us).
    // Taps and rows stay compile-time: run-time loops over them were measured slower (450-470 us; the set-up between the
    // hand-over and the first MMA is what the tensor pipe waits for)
#pragma unroll 1
    for (int k = K0; k < K1; k++) {
        const uint64_t da = desc64(a_lo + (uint32_t)(k * 2), DESC_HI_SW128);
#pragma unroll
        for (int r = ra; r < rb; r++) {
            const int sr = r + dy;
            const int cell0 = sr * BCOLS + (dx > 0 ? 1 : 0);
            const uint32_t boff = KMAJOR ? (uint32_t)((cell0 * (G * 128) + k * 32) >> 4) : (uint32_t)((k * 2 * KG_BYTES + cell0 * (G * 16)) >> 4);
            const uint32_t d = tbase + (uint32_t)(unit_of(r) * UNIT_COLS + (dx < 0 ? G : 0));
            const uint64_t db = desc64(b_lo + boff, KMAJOR ? DESC_HI_SW128 : DESC_HI_T16);
            const uint32_t acc = (k == 0 && first_touch(PASS, TI, r)) ? acc_first : 1u;
            // the rows share the weight tile: it is read from shared memory for the first one only
            if (rb - ra == 1) umma_bf16_coll<COLL_DISCARD>(d, da, db, idesc, acc);
            else if (r == ra) umma_bf16_coll<COLL_FILL>(d, da, db, idesc, acc);
            else if (r == rb - 1) umma_bf16_coll<COLL_LASTUSE>(d, da, db, idesc, acc);
            else umma_bf16_coll<COLL_USE>(d, da, db, idesc, acc);
        }
    }
}

// Two issuer warps (warp 1: even stages, warp 12: odd stages of the CTA's running stage count) take turns:
// the MMA queue of the tensor pipe is shallow, so with ONE issuer the pipe drains during every barrier wait,
// commit and loop step between stages (about a third of the time).  With two, warp B waits for the weights of
// stage s+1 while warp A's MMAs of stage s execute, and starts issuing the moment A hands over (named barrier;
// the hand-over comes after A's last MMA of the stage, so the A-operand collector groups never interleave).
// tcgen05 operations of one CTA execute in issue order, so accumulation order and the commits' coverage are
// those of the single-issuer sequence.  Each turn is one stage: what the second issuer buys is a warp that already
// waits for the NEXT stage's weights, and longer turns give that up (2 stages per turn: 416 us against 394).
__device__ __forceinline__ void named_bar_sync(int id) { asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void named_bar_arrive(int id) { asm volatile("bar.arrive %0, 64;" ::"r"(id) : "memory"); }

template <bool KMAJOR, int PASS, int TI>
struct StageLoop {
    // runs stages TI..8 of a pass for one channel half; each stage is issued by the warp whose parity matches
    template <class Ctx>
    static __device__ __forceinline__ void run(Ctx& c, int kh, int it, bool last_kh) {
        constexpr int NT = seg_nt(PASS);
        constexpr int r0 = seg_r0(PASS), r1 = seg_r1(PASS);
        if ((c.nstage & 1) == c.parity) {
            HZ_CTRACE(16 + 3 * c.nstage);
            mbar_wait(c.bar0 + 8u * (B_WFULL + c.stage), c.ph, c.fault, 0x400 + c.stage);
            if (kh == 0) {   // first touch of a row's accumulator for this tile: the unit's previous tenant must be drained
#pragma unroll
                for (int r = r0; r < r1; r++)
                    if (first_touch(PASS, TI, r)) mbar_wait(c.bar0 + 8u * (B_TEMPTY + unit_of(r)), (use_of(r, it) & 1) ^ 1, c.fault, 0x500 + r);
            }
            // everything the first MMA needs is computed before the hand-over is awaited
            const bool lead = elect_one();
            const uint32_t a_lo = DESC_LO_SW128 | ((c.sW + c.stage * W_BYTES) >> 4);
            const uint32_t b_lo = (KMAJOR ? DESC_LO_SW128 : DESC_LO_T16) | ((c.sX + (uint32_t)kh * KH_BYTES) >> 4);
            const uint32_t acc0 = kh == 0 ? 0u : 1u;
            if (c.nstage > 0) named_bar_sync(c.parity ? 1 : 2);   // the other issuer has handed over
            tc_fence_after();
            HZ_CTRACE(16 + 3 * c.nstage + 1);
            // (handing over BEFORE the last k-step, with that step issued without collector hints, was measured: the
            // interleaved MMAs corrupt the other issuer's collector group — results differ — so the hand-over stays behind
            // the last MMA; the commits, which only track this thread's own MMAs, come after it)
            if (lead && !(c.dbg & 1)) issue_stage<KMAJOR, PASS, TI, 0, 4>(a_lo, b_lo, c.tbase, acc0);
            __syncwarp();
            named_bar_arrive(c.parity ? 2 : 1);
            if (lead) {
                // frees the weight stage when these MMAs have read it (cluster mode: in every CTA of the cluster; the multicast
                // form with a mask of 1 in a launch without clusters was tried to save the branch: it faults)
                if (c.pair) umma_commit_mc(c.bar0 + 8u * (B_WEMPTY + c.stage), c.cmask);
                else umma_commit(c.bar0 + 8u * (B_WEMPTY + c.stage));
                if (last_kh) {
#pragma unroll
                    for (int r = r0; r < r1; r++)
                        if (last_touch(PASS, TI, r)) umma_commit(c.bar0 + 8u * (B_TFULL + unit_of(r)));
                }
                if (PASS == NSEG - 1 && TI == NT - 1) umma_commit(c.bar0 + 8u * (B_AEMPTY + kh));   // the tile's channel half is no longer read
            }
            __syncwarp();
            HZ_CTRACE(16 + 3 * c.nstage + 2);
        }
        c.nstage++;
        if (++c.stage == NSTAGE) { c.stage = 0; c.ph ^= 1; }
        if constexpr (TI < NT - 1) StageLoop<KMAJOR, PASS, TI + 1>::run(c, kh, it, last_kh);
    }
};

// the head item's stages: one tap (dy = dx = 0) over the rows {0,1,2} then {3,4}, per channel half; same protocol as StageLoop
template <int HSEG>
struct HeadStage {
    template <class Ctx>
    static __device__ __forceinline__ void run(Ctx& c, int kh, int it, bool last_kh) {
        constexpr int r0 = HSEG ? 3 : 0, r1 = HSEG ? 5 : 3;
        if ((c.nstage & 1) == c.parity) {
            mbar_wait(c.bar0 + 8u * (B_WFULL + c.stage), c.ph, c.fault, 0x400 + c.stage);
            if (kh == 0) {
#pragma unroll
                for (int r = r0; r < r1; r++) mbar_wait(c.bar0 + 8u * (B_TEMPTY + unit_of(r)), (use_of(r, it) & 1) ^ 1, c.fault, 0x500 + r);
            }
            const bool lead = elect_one();
            const uint32_t a_lo = DESC_LO_SW128 | ((c.sW + c.stage * W_BYTES) >> 4);
            const uint32_t b_lo = DESC_LO_T16 | ((c.sX + (uint32_t)kh * KH_BYTES) >> 4);
            const uint32_t acc0 = kh == 0 ? 0u : 1u;
            if (c.nstage > 0) named_bar_sync(c.parity ? 1 : 2);
            tc_fence_after();
            if (lead && !(c.dbg & 1)) {
                constexpr uint32_t idesc = idesc_bf16_f32(128, 112) | (1u << 16);
#pragma unroll 1
                for (int k = 0; k < 4; k++) {
                    const uint64_t da = desc64(a_lo + (uint32_t)(k * 2), DESC_HI_SW128);
#pragma unroll
                    for (int r = r0; r < r1; r++) {
                        const uint32_t boff = (uint32_t)((k * 2 * KG_BYTES + r * BCOLS * (G * 16)) >> 4);
                        const uint32_t d = c.tbase + (uint32_t)(unit_of(r) * UNIT_COLS);
                        const uint64_t db = desc64(b_lo + boff, DESC_HI_T16);
                        const uint32_t acc = k == 0 ? acc0 : 1u;
                        if (r == r0) umma_bf16_coll<COLL_FILL>(d, da, db, idesc, acc);
                        else if (r == r1 - 1) umma_bf16_coll<COLL_LASTUSE>(d, da, db, idesc, acc);
                        else umma_bf16_coll<COLL_USE>(d, da, db, idesc, acc);
                    }
                }
            }
            __syncwarp();
            named_bar_arrive(c.parity ? 2 : 1);
            if (lead) {
                if (c.pair) umma_commit_mc(c.bar0 + 8u * (B_WEMPTY + c.stage), c.cmask);
                else umma_commit(c.bar0 + 8u * (B_WEMPTY + c.stage));
                if (last_kh) {
#pragma unroll
                    for (int r = r0; r < r1; r++) umma_commit(c.bar0 + 8u * (B_TFULL + unit_of(r)));
                }
                if (HSEG == 1) umma_commit(c.bar0 + 8u * (B_AEMPTY + kh));
            }
            __syncwarp();
        }
        c.nstage++;
        if (++c.stage == NSTAGE) { c.stage = 0; c.ph ^= 1; }
    }
};

struct IssueCtx {
    uint32_t bar0, sW, sX, tbase, stage, ph;
    unsigned int* fault;
    int dbg;
    unsigned long long* trace;   // null unless CTA 0 is being traced
    int nstage;                  // running stage count of the CTA (turn and trace index)
    int parity;                  // this warp issues the stages with nstage % 2 == parity
    bool pair;                   // cluster mode: weight stages are shared with the other CTAs of the cluster
    uint16_t cmask;              // ... their mask
};

__device__ __forceinline__ unsigned int ld_acquire_gpu(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned int atom_add_acq_rel_gpu(unsigned int* p, unsigned int v) {
    unsigned int old;
    asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
    return old;
}
__device__ __forceinline__ void st_release_gpu(unsigned int* p, unsigned int v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// take the next ready item: slot = head++; the slot is filled (item + 1) by the CTA that completes the item's input
__device__ __forceinline__ int dequeue_item(unsigned int* sched, int n_items, unsigned int* fault) {
    const unsigned int slot = atomicAdd(sched, 1u);
    if (slot >= (unsigned int)n_items) return -1;
    const unsigned int* q = sched + 2 + n_items + slot;
    unsigned int v;
    for (uint32_t it = 0; (v = ld_acquire_gpu(q)) == 0u; ++it) {
        __nanosleep(64);
        if (it > (1u << 22)) {
            if (fault) { atomicExch(fault, 0xB00u); __threadfence_system(); }
            __trap();
        }
    }
    return (int)v - 1;
}

__global__ void __launch_bounds__(NTHREADS, 1) k_tower(const __grid_constant__ Params P) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* sm = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const uint32_t sX = smem_u32(sm + OFF_X), sW = smem_u32(sm + OFF_W), sBar = smem_u32(sm + OFF_BAR);
    uint32_t* tmem_slot = (uint32_t*)(sm + OFF_BAR + N_BARS * 8);
    volatile int* qitem = (volatile int*)(sm + OFF_BAR + N_BARS * 8 + 16);   // work-item queue, 2 entries
    auto bar = [&](int i) { return sBar + 8u * (uint32_t)i; };
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int crank = P.pair ? (int)cluster_ctarank() : 0;     // rank inside the cluster of two (pair mode)
    if (threadIdx.x == 0) {
        // pair mode: a weight stage is free again when the MMAs of BOTH CTAs have read it (each CTA's copies land in both)
        for (int i = 0; i < NSTAGE; i++) { mbar_init(bar(B_WFULL + i), 1); mbar_init(bar(B_WEMPTY + i), P.pair ? P.pair : 1); }
        for (int i = 0; i < 2; i++) { mbar_init(bar(B_AFULL + i), 1); mbar_init(bar(B_AEMPTY + i), 1); }
        for (int i = 0; i < NUNIT; i++) { mbar_init(bar(B_TFULL + i), 1); mbar_init(bar(B_TEMPTY + i), 8); }
        mbar_init(bar(B_DONE), 2);
        for (int i = 0; i < 2; i++) { mbar_init(bar(B_QFULL + i), 1); mbar_init(bar(B_QEMPTY + i), N_CONSUMERS); }
        mbar_init_fence();
    }
    if (warp == 3) tmem_alloc(smem_u32(tmem_slot), 512);
    tc_fence_before();
    __syncthreads();
    if (P.pair) cluster_sync_all();          // the peer's barriers exist before anything of ours can arrive on them
    tc_fence_after();
    const uint32_t tbase = *tmem_slot;
    const int n_tiles = tiles_of(P.n_active, P.n_tiles);
    const int csize = P.pair ? P.pair : 1;                       // CTAs per cluster = tiles per work unit (1, 2 or 4)
    const int n_units = (n_tiles + csize - 1) / csize;           // work units per layer: tiles, or groups of neighbouring tiles
    const int n_items = P.n_layers * n_units;
    // this CTA's tile of work unit u (an odd tile count makes both CTAs of the last pair compute the same tile)
    auto tile_of = [&](int u) { return min(csize * u + crank, n_tiles - 1); };
    if (warp == 0) HZ_TRACE(0);
    if (HZ_TOWER_TRACE && warp == 0 && P.trace && blockIdx.x == 0 && lane == 0) P.trace[2] = globaltimer_ns();

    // every role walks the CTA's work items in the order the scheduler (warp 3) publishes them; -1 ends the walk.
    // NEXT_ITEM: whole-warp roles call it converged; single-lane roles call it from their one lane.
#define HZ_NEXT_ITEM(k, item, whole_warp)                                                      \
    do {                                                                                       \
        mbar_wait(bar(B_QFULL + ((k) & 1)), ((uint32_t)(k) >> 1) & 1u, P.fault, 0x900 + warp); \
        item = qitem[(k) & 1];                                                                 \
        if (whole_warp) __syncwarp();                                                          \
        if (!(whole_warp) || lane == 0) mbar_arrive(bar(B_QEMPTY + ((k) & 1)));                \
        (k)++;                                                                                 \
    } while (0)

    if (warp == 3) {
        // ---- scheduler ----
        if (lane == 0) {
            const int per_cta = (n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // static map: tiles blockIdx.x + j*gridDim.x
            unsigned int* mbox = P.pair ? P.mailbox + (size_t)(blockIdx.x / (unsigned)P.pair) * 64 : nullptr;
            for (int k = 0;; k++) {
                int item;
                if (P.pair && crank != 0) {
                    // the item CTA 0 of this cluster drew as its k-th: entry = tag(k) << 20 | item + 2
                    const unsigned int want = (unsigned int)(k % 4095 + 1) << 20;     // never 0: a cleared mailbox matches nothing
                    unsigned int v;
                    for (uint32_t it = 0; ((v = ld_acquire_gpu(mbox + (k & 63))) & 0xFFF00000u) != want; ++it) {
                        __nanosleep(32);
                        if (it > (1u << 22)) {
                            if (P.fault) { atomicExch(P.fault, 0xB01u); __threadfence_system(); }
                            __trap();
                        }
                    }
                    item = (int)(v & 0xFFFFFu) - 2;
                } else if (P.sched) {
                    item = dequeue_item(P.sched, n_items, P.fault);
                    if (P.pair) st_release_gpu(mbox + (k & 63), ((unsigned int)(k % 4095 + 1) << 20) | (unsigned int)(item + 2));
                } else {
                    item = k < per_cta * P.n_layers ? (k / per_cta) * n_tiles + (int)blockIdx.x + (k % per_cta) * (int)gridDim.x : -1;
                }
                mbar_wait(bar(B_QEMPTY + (k & 1)), (((uint32_t)k >> 1) & 1u) ^ 1u, P.fault, 0xA00);
                qitem[k & 1] = item;
                mbar_arrive(bar(B_QFULL + (k & 1)));      // release: the consumers' waits acquire the slot
                if (item < 0) break;
            }
        }
    } else if (warp == 0) {
        // ---- weight producer: the tap stream of every pass of every item, through the ring ----
        if (lane == 0) {
            uint32_t stage = 0, ph = 0;
            int ns = 0, k = 0;
            for (;;) {
                int item;
                HZ_NEXT_ITEM(k, item, false);
                if (item < 0) break;
                const Layer& L = P.layers[item / n_units];
                const int nkh = L.nkh;
                const int nseg = L.head ? 2 : NSEG;
                for (int seg = 0; seg < nseg; seg++)
                    for (int kh = 0; kh < nkh; kh++)
                        for (int ti = 0; ti < (L.head ? 1 : seg_nt(seg)); ti++, ns++) {
                            int tap = L.head ? 0 : SEG_TAPS[seg][ti];
                            mbar_wait(bar(B_WEMPTY + stage), ph ^ 1, P.fault, 0x100 + stage);
                            if (ns < 600) { HZ_TRACE(2000 + ns); }
                            if (P.dbg & 4) mbar_arrive(bar(B_WFULL + stage));
                            else {
                                mbar_expect_tx(bar(B_WFULL + stage), W_BYTES);
                                const uint8_t* wsrc = L.w + (size_t)(tap * nkh + kh) * W_BYTES;
                                if (P.pair) {   // this CTA's share of the stage, delivered to every CTA of the cluster
                                    const uint32_t part = W_BYTES / (uint32_t)P.pair;
                                    bulk_g2s_mc(sW + stage * W_BYTES + crank * part, wsrc + crank * part, part, bar(B_WFULL + stage),
                                                (uint16_t)((1u << P.pair) - 1u));
                                }
                                else bulk_g2s(sW + stage * W_BYTES, wsrc, W_BYTES, bar(B_WFULL + stage));
                            }
                            if (++stage == NSTAGE) { stage = 0; ph ^= 1; }
                        }
            }
        }
    } else if (warp == 2) {
        // ---- activation producer: one channel half of a tile per buffer ----
        if (lane == 0) {
            uint32_t cnt0 = 0, cnt1 = 0;       // uses of each half buffer so far (barrier phase)
            int na = 0, k = 0;
            for (;;) {
                int item;
                HZ_NEXT_ITEM(k, item, false);
                if (item < 0) break;
                const int l = item / n_units, tile = tile_of(item - l * n_units);
                const Layer& L = P.layers[l];
                // the tile's input is the previous layer's output, possibly written by another CTA through the generic
                // proxy; the ready queue (acquired by the scheduler, handed over through the item barrier) makes it
                // visible to this thread, the proxy fence orders the async-proxy reads behind that
                if (l > 0) fence_proxy_async();
                for (int kh = 0; kh < L.nkh; kh++, na++) {
                    mbar_wait(bar(B_AEMPTY + kh), ((kh ? cnt1 : cnt0) & 1u) ^ 1u, P.fault, 0x200 + kh);
                    if (kh) cnt1++; else cnt0++;
                    if (na < 400) { HZ_TRACE(3600 + na); }
                    if (P.dbg & 8) { mbar_arrive(bar(B_AFULL + kh)); continue; }
                    mbar_expect_tx(bar(B_AFULL + kh), KH_BYTES);
                    const uint8_t* src = P.buf[L.in_buf] + ((size_t)tile * L.nkh + kh) * KH_BYTES;
                    for (int r = 0; r < BROWS; r++)
                        bulk_g2s(sX + kh * KH_BYTES + r * ROW_BYTES, src + (size_t)r * ROW_BYTES, ROW_BYTES, bar(B_AFULL + kh));
                }
            }
        }
    } else if (warp == 1 || warp == 12) {
        // ---- MMA issuers: the whole warp runs the loop, one elected lane issues its stages ----
        IssueCtx c{sBar, sW, sX, tbase, 0u, 0u, P.fault, P.dbg, (blockIdx.x == 0 && lane == 0) ? P.trace : nullptr, 0, warp == 12 ? 1 : 0, P.pair != 0, (uint16_t)((1u << (P.pair ? P.pair : 1)) - 1u)};
        uint32_t cnt0 = 0, cnt1 = 0;
        int wi = 0, k = 0;                 // wi: work items done (phase of the accumulator units)
        for (;; wi++) {
            int item;
            HZ_NEXT_ITEM(k, item, true);
            if (item < 0) break;
            const Layer& L = P.layers[item / n_units];
            const int nkh = L.nkh;
            const bool kmajor = L.kmajor != 0;
            if (L.head) {
                for (int kh = 0; kh < nkh; kh++) {
                    mbar_wait(bar(B_AFULL + kh), (kh ? cnt1 : cnt0) & 1u, P.fault, 0x300 + kh);
                    if (kh) cnt1++; else cnt0++;
                    HeadStage<0>::run(c, kh, wi, kh == nkh - 1);
                }
                for (int kh = 0; kh < nkh; kh++) HeadStage<1>::run(c, kh, wi, kh == nkh - 1);
                continue;
            }
            for (int kh = 0; kh < nkh; kh++) {
                mbar_wait(bar(B_AFULL + kh), (kh ? cnt1 : cnt0) & 1u, P.fault, 0x300 + kh);   // both issuers observe the tile half
                if (kh) cnt1++; else cnt0++;
                if (kmajor) StageLoop<true, 0, 0>::run(c, kh, wi, kh == nkh - 1);
                else StageLoop<false, 0, 0>::run(c, kh, wi, kh == nkh - 1);
            }
            for (int kh = 0; kh < nkh; kh++) {
                if (kmajor) StageLoop<true, 1, 0>::run(c, kh, wi, kh == nkh - 1);
                else StageLoop<false, 1, 0>::run(c, kh, wi, kh == nkh - 1);
            }
        }
        // the last hand-over has no taker yet: the warp whose turn would be next consumes it
        if (c.nstage > 0 && (c.nstage & 1) == c.parity) named_bar_sync(c.parity ? 1 : 2);
        if (elect_one()) umma_commit(bar(B_DONE));
        __syncwarp();
        mbar_wait(bar(B_DONE), 0, P.fault, 0x600);
    } else if (warp >= 4 && warp < 12) {
        // ---- epilogue: 8 warps.  thread = output channel c (TMEM lane); warps 4-7 take cells x = 0..3
        // of a board row, warps 8-11 cells x = 4..6.  One TMEM load = the 16 boards of a cell = 2 x 16
        // contiguous bytes of channel c's row in the T16 image (vector stores, vector residual loads).
        // All TMEM loads of the row are issued back to back and the unit is released as soon as they
        // have landed in registers, before the arithmetic and the stores.
        const int q = warp & 3, c = q * 32 + lane;
        const int half = (warp - 4) >> 2;
        const int x0 = half ? 4 : 0;
        const uint32_t chan_off = (uint32_t)(c >> 3) * KG_BYTES + (uint32_t)(c & 7) * 16u;
        const bool mem = !(P.dbg & 2);
        int nrow = 0, k = 0;
        for (int wi = 0;; wi++) {
            int item;
            HZ_NEXT_ITEM(k, item, true);
            if (item < 0) break;
            const int l = item / n_units, tile = tile_of(item - l * n_units);
            const Layer& L = P.layers[l];
            if (L.head) {
                // head item: output filter j = accumulator lanes j (high part) and j + 3 (low part): only the first warp of
                // each cell half has data; every warp keeps the accumulator protocol
                const float hbias = (q == 0 && lane < 3) ? L.bias[lane] : 0.0f;
                float* hout = L.head_out + (size_t)tile * (3 * CELLS * G);
                for (int ri = 0; ri < BROWS; ri++, nrow++) {
                    const int r = EPI_ORDER[ri], unit = unit_of(r);
                    mbar_wait(bar(B_TFULL + unit), use_of(r, wi) & 1, P.fault, 0x700 + unit);
                    tc_fence_after();
                    if (q == 0) {
                        // one cell at a time (16 registers): the head item is short, register pressure here must not
                        // spill the convolution epilogue below
                        const uint32_t ta = tbase + unit * UNIT_COLS + x0 * G;
#pragma unroll 1
                        for (int j = 0; j < (half ? 3 : 4); j++) {
                            uint32_t v[16];
                            tmem_ld16(ta + j * G, v);
                            tmem_ld_wait();
                            float o[16];
#pragma unroll
                            for (int b = 0; b < G; b++) {
                                const float hi = __uint_as_float(v[b]);
                                o[b] = fmaxf(hi + __shfl_down_sync(0xFFFFFFFFu, hi, 3) + hbias, 0.0f);
                            }
                            if (lane < 3 && mem) {
                                float4* dst = reinterpret_cast<float4*>(hout + ((size_t)lane * CELLS + (r * BCOLS + x0 + j)) * G);
#pragma unroll
                                for (int e = 0; e < 4; e++) dst[e] = make_float4(o[4 * e], o[4 * e + 1], o[4 * e + 2], o[4 * e + 3]);
                            }
                        }
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar(B_TEMPTY + unit));
                }
                continue;
            }
            const float bias = L.bias[c];
            const uint8_t* resb = (L.res_buf >= 0 && mem) ? P.buf[L.res_buf] : nullptr;
            uint8_t* yb = P.buf[L.out_buf];
            const bool relu = L.relu != 0;
            // (the residual — the block input, two layers back, possibly written by another CTA — is visible: every hand-over
            // of this tile went through a gpu-scope release/acquire of the ready queue and this CTA's item barrier)
            const size_t tile_off = (size_t)tile * 2 * KH_BYTES + chan_off;
            for (int ri = 0; ri < BROWS; ri++, nrow++) {
                const int r = EPI_ORDER[ri], unit = unit_of(r);
                const size_t row_off = tile_off + (size_t)(r * BCOLS + x0) * (G * 16);
                // the residual of this warp's cells is requested before the accumulator is waited for
                uint4 rv[8];
                if (resb) {
#pragma unroll
                    for (int j = 0; j < 4; j++)
                        if (j < 3 || !half) {
                            const uint8_t* rp = resb + row_off + (size_t)j * (G * 16);
                            rv[2 * j] = *reinterpret_cast<const uint4*>(rp);
                            rv[2 * j + 1] = *reinterpret_cast<const uint4*>(rp + 128);
                        }
                }
                if (warp == 4 && nrow < 200) { HZ_TRACE(2700 + 4 * nrow); }
                mbar_wait(bar(B_TFULL + unit), use_of(r, wi) & 1, P.fault, 0x700 + unit);
                tc_fence_after();
                if (warp == 4 && nrow < 200) { HZ_TRACE(2700 + 4 * nrow + 1); }
                uint32_t v[4][16];
                const uint32_t ta = tbase + ((uint32_t)(q * 32) << 16) + unit * UNIT_COLS + x0 * G;
                tmem_ld16(ta, v[0]);
                tmem_ld16(ta + G, v[1]);
                tmem_ld16(ta + 2 * G, v[2]);
                if (!half) tmem_ld16(ta + 3 * G, v[3]);
                tmem_ld_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar(B_TEMPTY + unit));      // the accumulator may be overwritten from here on
                if (warp == 4 && nrow < 200) { HZ_TRACE(2700 + 4 * nrow + 2); }
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    if (j == 3 && half) break;
                    float o[16];
#pragma unroll
                    for (int b = 0; b < G; b++) o[b] = __uint_as_float(v[j][b]) + bias;
                    if (resb) {
                        const uint32_t* rw = reinterpret_cast<const uint32_t*>(&rv[2 * j]);
#pragma unroll
                        for (int e = 0; e < 8; e++) {
                            o[2 * e] += __uint_as_float(rw[e] << 16);
                            o[2 * e + 1] += __uint_as_float(rw[e] & 0xFFFF0000u);
                        }
                    }
                    uint8_t* yp = yb + row_off + (size_t)j * (G * 16);
                    if (!mem) { if (o[0] + o[5] + o[10] + o[15] == 12345.678f) *reinterpret_cast<float*>(yp) = o[3]; continue; }
                    uint32_t pk[8];
                    if (relu) {
#pragma unroll
                        for (int e = 0; e < 8; e++) pk[e] = pack_bf16x2_relu(o[2 * e], o[2 * e + 1]);
                    } else {
#pragma unroll
                        for (int e = 0; e < 8; e++) pk[e] = pack_bf16x2(o[2 * e], o[2 * e + 1]);
                    }
                    *reinterpret_cast<uint4*>(yp) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                    *reinterpret_cast<uint4*>(yp + 128) = make_uint4(pk[4], pk[5], pk[6], pk[7]);
                }
                if (warp == 4 && nrow < 200) { HZ_TRACE(2700 + 4 * nrow + 3); }
            }
            if (P.sched && l + 1 < P.n_layers) {
                // publish the tile's output: generic-proxy stores -> visible at gpu scope and to async-proxy readers
                __threadfence();
                fence_proxy_async();
                __syncwarp();
                unsigned int last = 0;
                if (lane == 0) last = atom_add_acq_rel_gpu(P.sched + 2 + item, 1u) == (unsigned)csize * FLAG_DONE - 1 ? 1u : 0u;
                last = __shfl_sync(0xFFFFFFFFu, last, 0);
                if (last) {
                    // last of the 8 epilogue warps to finish the item
                    // the tile's next layer becomes ready
                    if (lane == 0) {
                        const unsigned int slot = atomicAdd(P.sched + 1, 1u);
                        st_release_gpu(P.sched + 2 + n_items + slot, (unsigned int)(item + n_units) + 1u);
                    }
                }
            }
        }
    }
#undef HZ_NEXT_ITEM
    tc_fence_before();
    __syncthreads();
    if (P.pair) cluster_sync_all();          // neither CTA leaves while the other may still deliver weights or commits to it
    if (warp == 0) HZ_TRACE(1);
    if (HZ_TOWER_TRACE && warp == 0 && P.trace && blockIdx.x == 0 && lane == 0) P.trace[3] = globaltimer_ns();
    if (warp == 3) tmem_dealloc(tbase, 512);
}

// ready queue before the launch: head 0, tail n_tiles, no completions, the stem items in slots 0..n_tiles-1
constexpr int MAILBOX_WORDS = 128 * 64;     // pair mode: 64 words per cluster
__global__ void k_sched_init(unsigned int* sched, int n_tiles_max, int n_layers, const int* n_active, int pair, unsigned int* mailbox) {
    const int n_tiles = tiles_of(n_active, n_tiles_max), n_units = pair ? (n_tiles + pair - 1) / pair : n_tiles, n_items = n_layers * n_units;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 2 + 2 * n_items; i += gridDim.x * blockDim.x) {
        unsigned int v = 0u;
        if (i == 1) v = (unsigned int)n_units;
        else if (i >= 2 + n_items && i < 2 + n_items + n_units) v = (unsigned int)(i - (2 + n_items)) + 1u;
        sched[i] = v;
    }
    if (mailbox)
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < MAILBOX_WORDS; i += gridDim.x * blockDim.x) mailbox[i] = 0u;
}

// ---- layout conversion (interop with NHWC tensors: tests, the heads kernel) -----------------------
// src [n][35][C] bf16 (C % 8 == 0, C <= 64) -> T16K tiles [n_pad/16][560][128 B]; pad boards/channels = 0
__global__ void k_to_tiles_k(const uint4* __restrict__ src, uint4* __restrict__ dst, int64_t n, int C, int64_t n_chunks) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_chunks; i += (int64_t)gridDim.x * blockDim.x) {
        int j = (int)(i & 7);                       // chunk position inside the 128-byte row (swizzled)
        int64_t row = i >> 3;                       // tile*560 + p
        int p = (int)(row % TILE_ROWS);
        int64_t tile = row / TILE_ROWS;
        int cell = p / G, b = p % G;
        int ch = (j ^ (p & 7)) * 8;                 // logical 8-channel group stored at position j
        int64_t board = tile * G + b;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (board < n && ch < C) v = src[((board * CELLS + cell) * C + ch) >> 3];
        dst[i] = v;
    }
}
// src [n][35][128] bf16 -> T16 tiles (2 halves); one thread = 8 positions of one channel (a 16-byte chunk)
__global__ void k_to_tiles(const __nv_bfloat16* __restrict__ src, uint4* __restrict__ dst, int64_t n, int64_t n_chunks) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_chunks; i += (int64_t)gridDim.x * blockDim.x) {
        int k8 = (int)(i & 7);
        int64_t g = i >> 3;                         // (tile*16 + kg)*70 + pg
        int pg = (int)(g % (TILE_ROWS / 8));
        int64_t tk = g / (TILE_ROWS / 8);
        int kg = (int)(tk & 15);
        int64_t tile = tk >> 4;
        int c = kg * 8 + k8;
        uint32_t w[4];
#pragma unroll
        for (int h = 0; h < 4; h++) {
            uint32_t two = 0;
#pragma unroll
            for (int e = 0; e < 2; e++) {
                int p = pg * 8 + 2 * h + e, cell = p / G;
                int64_t board = tile * G + p % G;
                uint32_t bits = board < n ? (uint32_t)__bfloat16_as_ushort(src[(board * CELLS + cell) * 128 + c]) : 0u;
                two |= bits << (16 * e);
            }
            w[h] = two;
        }
        dst[i] = make_uint4(w[0], w[1], w[2], w[3]);
    }
}
// T16 tiles (2 halves) -> dst [n][35][128] bf16; one thread = one output element pair
__global__ void k_from_tiles(const __nv_bfloat16* __restrict__ src, __nv_bfloat16* __restrict__ dst, int64_t n_elems) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_elems; i += (int64_t)gridDim.x * blockDim.x) {
        int c = (int)(i & 127);
        int64_t pos = i >> 7;                       // board*35 + cell
        int cell = (int)(pos % CELLS);
        int64_t board = pos / CELLS;
        int p = cell * G + (int)(board % G);
        size_t off = (size_t)(board / G) * 2 * KH_BYTES + (size_t)(c >> 3) * KG_BYTES + (size_t)(p >> 3) * 128 + (c & 7) * 16 + (p & 7) * 2;
        dst[i] = src[off >> 1];
    }
}

#define MAX_LAYERS_SCHED(n_blocks) (2 + 2 * (n_blocks))   /* layers hz_tower_sched_bytes reserves queue space for */
static int g_debug = 0;
static unsigned long long* g_trace = nullptr;
static int g_max_ctas = 0;   // 0 = one CTA per SM; tests lower it to drive several tiles through one CTA

static int ensure_attr() {
    static bool done[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !done[dev]) {
        cudaError_t e = cudaFuncSetAttribute(k_tower, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
        if (e != cudaSuccess) return hz_record_launch(0, e);
        if (dev >= 0 && dev < 64) done[dev] = true;
    }
    return HZ_OK;
}

static int grid_for(int n_tiles) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_max_ctas > 0 && g_max_ctas < sms) sms = g_max_ctas;
    return n_tiles < sms ? n_tiles : sms;
}

}  // namespace tower
}  // namespace hz

extern "C" {

size_t hz_tower_tile_bytes(int64_t n_boards, int channel_halves) {
    if (n_boards < 0 || channel_halves < 1 || channel_halves > 2) return 0;
    int64_t tiles = (n_boards + hz::tower::G - 1) / hz::tower::G;
    return (size_t)tiles * channel_halves * hz::tower::KH_BYTES;
}

int hz_tower_set_max_ctas(int max_ctas) {
    hz::tower::g_max_ctas = max_ctas > 0 ? max_ctas : 0;
    return HZ_OK;
}

int hz_tower_set_debug(int flags) {
    hz::tower::g_debug = flags;
    return HZ_OK;
}

int hz_tower_set_trace(unsigned long long* device_buffer_4096) {
    if (device_buffer_4096 && !HZ_TOWER_TRACE) return HZ_ERR_ARG;   // the time stamps are compiled in with -DHZ_TOWER_TRACE=1 only
    hz::tower::g_trace = device_buffer_4096;
    return HZ_OK;
}

int hz_tower_to_tiles(const void* src_nhwc, void* dst_tiles, int64_t n_boards, int channels, int kmajor, void* stream) {
    if (!src_nhwc || !dst_tiles || n_boards <= 0 || ((uintptr_t)src_nhwc & 15) || ((uintptr_t)dst_tiles & 15)) return HZ_ERR_ARG;
    if (kmajor ? (channels <= 0 || (channels & 7) || channels > 64) : channels != 128) return HZ_ERR_ARG;
    int64_t tiles = (n_boards + hz::tower::G - 1) / hz::tower::G;
    int64_t n_chunks = tiles * (kmajor ? 1 : 2) * hz::tower::TILE_ROWS * 8;
    int grid = (int)((n_chunks + 255) / 256 < 148 * 16 ? (n_chunks + 255) / 256 : 148 * 16);
    if (kmajor)
        hz::tower::k_to_tiles_k<<<grid, 256, 0, (cudaStream_t)stream>>>((const uint4*)src_nhwc, (uint4*)dst_tiles, n_boards, channels, n_chunks);
    else
        hz::tower::k_to_tiles<<<grid, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)src_nhwc, (uint4*)dst_tiles, n_boards, n_chunks);
    return hz_launched(1);
}

int hz_tower_from_tiles(const void* src_tiles, void* dst_nhwc, int64_t n_boards, void* stream) {
    if (!src_tiles || !dst_nhwc || n_boards <= 0 || ((uintptr_t)src_tiles & 15) || ((uintptr_t)dst_nhwc & 15)) return HZ_ERR_ARG;
    int64_t n_elems = n_boards * hz::tower::CELLS * 128;
    int grid = (int)((n_elems + 255) / 256 < 148 * 32 ? (n_elems + 255) / 256 : 148 * 32);
    hz::tower::k_from_tiles<<<grid, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)src_tiles, (__nv_bfloat16*)dst_nhwc, n_elems);
    return hz_launched(1);
}

int hz_tower_conv3x3(const void* x_tiles, int in_channel_halves, int in_kmajor, const void* w_tiles, const float* bias,
                     const void* residual_tiles, void* y, int64_t n_boards, int relu, unsigned int* fault, void* stream) {
    using namespace hz::tower;
    if (!x_tiles || !w_tiles || !bias || !y || n_boards <= 0 || (n_boards % G) || in_channel_halves < 1 || in_channel_halves > 2)
        return HZ_ERR_ARG;
    if (in_kmajor && in_channel_halves != 1) return HZ_ERR_ARG;
    if (((uintptr_t)x_tiles | (uintptr_t)w_tiles | (uintptr_t)y | (uintptr_t)residual_tiles) & 15) return HZ_ERR_ARG;
    int st = ensure_attr();
    if (st != HZ_OK) return st;
    Params P{};
    P.buf[0] = (uint8_t*)x_tiles;
    P.buf[1] = (uint8_t*)residual_tiles;
    P.buf[2] = (uint8_t*)y;
    P.layers[0] = Layer{(const uint8_t*)w_tiles, bias, 0, residual_tiles ? 1 : -1, 2, in_channel_halves, in_kmajor, relu};
    P.n_layers = 1;
    P.n_tiles = (int)(n_boards / G);
    P.sched = nullptr;
    P.fault = fault;
    P.dbg = g_debug;
    P.trace = g_trace;
    k_tower<<<grid_for(P.n_tiles), NTHREADS, SMEM_BYTES, (cudaStream_t)stream>>>(P);
    return hz_launched(1);
}

size_t hz_tower_sched_bytes(int64_t n_boards, int n_blocks) {
    if (n_boards <= 0 || n_blocks < 0) return 0;
    int64_t tiles = (n_boards + hz::tower::G - 1) / hz::tower::G;
    return sizeof(unsigned int) * ((size_t)(2 + 2 * (2 + 2 * n_blocks) * tiles) + hz::tower::MAILBOX_WORDS);   // + the optional head item per tile, + the pair-mode mailboxes
}

int hz_tower_forward_heads(const void* x0_tiles, const void* const* w_tiles, const float* const* biases, int n_blocks, void* buf_a,
                           void* buf_b, void* buf_c, void* sched, void** out_tiles, int64_t n_boards, const int32_t* n_active,
                           const void* w_head_tiles, const float* b_head, float* head_conv_tiled, unsigned int* fault, void* stream) {
    using namespace hz::tower;
    if ((uintptr_t)n_active & 3) return HZ_ERR_ARG;
    if (w_head_tiles && (!b_head || !head_conv_tiled || (((uintptr_t)w_head_tiles | (uintptr_t)head_conv_tiled) & 15) || 2 + 2 * n_blocks > MAX_LAYERS))
        return HZ_ERR_ARG;
    if (!x0_tiles || !w_tiles || !biases || !buf_a || !buf_b || !buf_c || !sched || n_boards <= 0 || (n_boards % G) || n_blocks < 0 ||
        1 + 2 * n_blocks > MAX_LAYERS)
        return HZ_ERR_ARG;
    if (((uintptr_t)x0_tiles | (uintptr_t)buf_a | (uintptr_t)buf_b | (uintptr_t)buf_c | (uintptr_t)sched) & 15) return HZ_ERR_ARG;
    int st = ensure_attr();
    if (st != HZ_OK) return st;
    Params P{};
    P.buf[0] = (uint8_t*)x0_tiles;
    P.buf[1] = (uint8_t*)buf_a;
    P.buf[2] = (uint8_t*)buf_b;
    P.buf[3] = (uint8_t*)buf_c;
    // stem: x0 -> a; block i: conv1 cur -> b, conv2 b (+ cur) -> nxt; cur and nxt alternate between a and c
    int n = 0, cur = 1, nxt = 3;
    for (int i = 0; i < 1 + 2 * n_blocks; i++)
        if (!w_tiles[i] || !biases[i] || ((uintptr_t)w_tiles[i] & 15)) return HZ_ERR_ARG;
    P.layers[n] = Layer{(const uint8_t*)w_tiles[0], biases[0], 0, -1, cur, 1, 1, 1};
    n++;
    for (int b = 0; b < n_blocks; b++) {
        P.layers[n] = Layer{(const uint8_t*)w_tiles[n], biases[n], cur, -1, 2, 2, 0, 1};
        n++;
        P.layers[n] = Layer{(const uint8_t*)w_tiles[n], biases[n], 2, cur, nxt, 2, 0, 1};
        n++;
        int t = cur; cur = nxt; nxt = t;
    }
    if (w_head_tiles) {
        P.layers[n] = Layer{(const uint8_t*)w_head_tiles, b_head, cur, -1, 0, 2, 0, 1, 1, head_conv_tiled};
        n++;
    }
    P.n_layers = n;
    P.n_tiles = (int)(n_boards / G);
    P.sched = (unsigned int*)sched;
    P.fault = fault;
    P.dbg = g_debug;
    P.trace = g_trace;
    P.n_active = n_active;
    if (out_tiles) *out_tiles = P.buf[cur];
    const int n_items = P.n_layers * P.n_tiles;
    // pair mode (clusters of two CTAs sharing the weight stream by multicast) unless there is a single tile or a single CTA
    P.pair = grid_for(P.n_tiles) >= 2 ? 2 : 0;
    P.mailbox = P.sched + (2 + 2 * (size_t)MAX_LAYERS_SCHED(n_blocks) * P.n_tiles);
    k_sched_init<<<(2 + 2 * n_items + 255) / 256, 256, 0, (cudaStream_t)stream>>>(P.sched, P.n_tiles, P.n_layers, n_active, P.pair, P.mailbox);
    if (P.pair) {
        const int n_units = (P.n_tiles + P.pair - 1) / P.pair;
        int clusters = grid_for(P.n_tiles) / P.pair;
        if (clusters > n_units) clusters = n_units;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(P.pair * clusters);
        cfg.blockDim = dim3(NTHREADS);
        cfg.dynamicSmemBytes = SMEM_BYTES;
        cfg.stream = (cudaStream_t)stream;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = P.pair; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
        cudaError_t e = cudaLaunchKernelEx(&cfg, k_tower, P);
        if (e != cudaSuccess) return hz_record_launch(1, e);
    } else {
        k_tower<<<grid_for(P.n_tiles), NTHREADS, SMEM_BYTES, (cudaStream_t)stream>>>(P);
    }
    return hz_launched(2);
}

}  // extern "C"
