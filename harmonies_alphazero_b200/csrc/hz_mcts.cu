// hz_mcts.cu — flat-array search trees (sm_100a): one warp owns one tree (one game), all
// trees advance one simulation per kernel pair (select -> [network] -> expand+backup).
//
// Replaces MCTS.py's per-game Python objects (Node/Edge/MCTS, MCTS.py:8-61) with per-tree
// arenas in caller-owned HBM:
//   nodes : packed 128 B states (AoS: a gather of one node is one full cache line), 64-bit
//           keys, first-edge index, edge count, player
//   edges : SoA child / N / W(fp64) / P(fp32) / (action | mover<<8); a node's edges are
//           contiguous and in ascending action order, so a warp reads them coalesced and
//           "first strict maximum" (MCTS.py:102,118) is a lowest-lane tie-break
//   table : open-addressing hash set (node index + 1) keyed by the 64-bit canonical key;
//           identity = key equality, as the reference's dict of hash(state) ids
//           (MCTS.py:184-186; -DHZ_TREE_FULL_COMPARE=1 adds a 23-word compare on hits)
// Parity mode is one in-flight simulation per tree (the reference is strictly sequential,
// MCTS.py:291-352); parallelism comes from thousands of concurrent trees.
#include <math.h>
#include <stdlib.h>

#include "hz_common.cuh"
#include "hz_core.cuh"
#include "hz_sym.cuh"

struct hz_tree {
    int n_trees, max_sims, max_nodes, max_edges, table_size, key_mode;
    int leaves;             // K simulations in flight per tree and step (1 = the reference's sequential search)
    uint4* node_state;      // [n_trees * max_nodes * 8]
    uint64_t* node_hash;    // [n_trees * max_nodes]
    uint32_t* node_edge0;   // [n_trees * max_nodes]
    uint32_t* node_info;    // [n_trees * max_nodes]  n_edges | player << 8 (| frame << 16 under hz_tree_set_symmetry)
    uint32_t* edge_child;   // [n_trees * max_edges]
    int32_t* edge_N;
    double* edge_W;
    float* edge_P;
    uint16_t* edge_am;      // action | mover << 8
    int32_t* edge_V;        // in-flight (virtual-loss) visits, non-zero only between select and backup
    uint32_t* edge_cinfo;   // cached (first edge | edge count << 24) of the child once it is known to be expanded, else 0
    uint32_t* table;        // [n_trees * table_size]  node index + 1, 0 = empty
    uint64_t* table_hash;   // [n_trees * table_size]  key of that node (valid where table != 0): a probe is ONE round trip
    uint32_t* path;         // [n_trees * leaves * (max_sims + 1)]
    int32_t* depth;         // [n_trees * leaves]
    int32_t* leaf;          // [n_trees * leaves]
    int32_t* sim;
    int32_t* n_nodes;
    int32_t* n_edges;
    uint8_t* status;
    uint64_t* search_key;
    size_t table_bytes;
    const int32_t* n_active;   // device word (nullable): only trees 0..*n_active-1 take part in reset / select / evaluate / expand
    int sym_mode;           // HZ_SYM_* of the launches that follow (hz_tree_set_symmetry)
    int frames_on;          // host side: the last hz_tree_select ran with a mode on
};

namespace hz {

constexpr int WPB = 4;            // warps (trees) per block
constexpr int TTPB = WPB * 32;
constexpr unsigned FULL = 0xFFFFFFFFu;

// trees beyond the active prefix (hz_tree_set_active) are skipped by the per-simulation kernels
__device__ __forceinline__ int active_trees(const hz_tree& T) {
    if (!T.n_active) return T.n_trees;
    int n = *T.n_active;
    return n < 0 ? 0 : n < T.n_trees ? n : T.n_trees;
}

struct TreeView {                 // device copy of the handle with per-tree offsets applied
    uint4* node_state; uint64_t* node_hash; uint32_t* node_edge0; uint32_t* node_info;
    uint32_t* edge_child; int32_t* edge_N; double* edge_W; float* edge_P; uint16_t* edge_am; int32_t* edge_V;
    uint32_t* edge_cinfo; uint32_t* table; uint64_t* table_hash; uint32_t* path;   // path: [leaves][max_sims + 1]
};
__device__ __forceinline__ TreeView view_of(const hz_tree& T, int t) {
    TreeView v;
    size_t nb = (size_t)t * T.max_nodes, eb = (size_t)t * T.max_edges;
    v.node_state = T.node_state + nb * 8; v.node_hash = T.node_hash + nb;
    v.node_edge0 = T.node_edge0 + nb; v.node_info = T.node_info + nb;
    v.edge_child = T.edge_child + eb; v.edge_N = T.edge_N + eb; v.edge_W = T.edge_W + eb;
    v.edge_P = T.edge_P + eb; v.edge_am = T.edge_am + eb; v.edge_V = T.edge_V + eb;
    v.edge_cinfo = T.edge_cinfo + eb;
    v.table = T.table + (size_t)t * T.table_size;
    v.table_hash = T.table_hash + (size_t)t * T.table_size;
    v.path = T.path + (size_t)t * T.leaves * (T.max_sims + 1);
    return v;
}

// warp-cooperative load of one node's state into shared memory (one 128 B line)
__device__ __forceinline__ void warp_load_words(uint32_t* sm, const uint4* node_state, int node, int lane) {
    sm[lane] = reinterpret_cast<const uint32_t*>(node_state + (size_t)node * 8)[lane];
    __syncwarp();
}
__device__ __forceinline__ void state_from_words(State& s, const uint32_t* sm) {
#pragma unroll
    for (int i = 0; i < SW; i++) s.w[i] = sm[i];
}

// ---- reset: Node(root) + MCTS(root) (MCTS.py:288-289, 43-61) -----------------------------------
__global__ void __launch_bounds__(TTPB) k_tree_reset(hz_tree T, const uint4* roots, const uint64_t* keys) {
    int t = blockIdx.x * TTPB + threadIdx.x;
    if (t >= active_trees(T)) return;
    TreeView v = view_of(T, t);
    State s;
    load_state(s, roots, t);
    store_state(s, v.node_state, 0);
    uint64_t h = canon_hash(s, T.key_mode);
    v.node_hash[0] = h;
    v.node_edge0[0] = 0;
    v.node_info[0] = (uint32_t)player_of(s) << 8;
    v.table[h & (uint64_t)(T.table_size - 1)] = 1;
    v.table_hash[h & (uint64_t)(T.table_size - 1)] = h;
    for (int j = 0; j < T.leaves; j++) { T.depth[t * T.leaves + j] = 0; T.leaf[t * T.leaves + j] = 0; }
    T.sim[t] = 0; T.n_nodes[t] = 1; T.n_edges[t] = 0;
    // a reset starts a new search but must not erase the record of a truncated one: the flags of
    // the search that ends here move to the sticky high nibble (cleared only by hz_tree_create)
    { uint8_t s8 = T.status[t]; T.status[t] = (uint8_t)((s8 & 0xF0u) | ((s8 & 0x0Fu) << 4)); }
    // default key: a stream of its own per (game, move), independent of the game's draw stream
    T.search_key[t] = keys ? keys[t] : rand64(key_of(s) ^ HZ_SEARCH_SALT, (uint64_t)s.w[HZ_W_MOVES]);
}

// Fast leaf encoder for the self-play layout (bf16, NHWC40): the 40 channels of a cell are
// 5 bytes of bits (<= 3+3 tile codes + player + phase), and 8 bits expand to a 16-byte vector
// of bf16 0.0/1.0 by one table lookup: 35 cells x 5 vectors = 175 16-byte stores per leaf
// instead of 1,400 scalar ones.
// T16K = true: the 16-byte groups go straight into the stem's tensor-core operand image
// (include/harmonies_b200.h "T16K": tile of 16 leaves, row p = cell*16 + leaf, group j at j ^ (p & 7));
// groups 5..7 (channels 40..63) of a row are never written and must have been zeroed once.
template <bool T16K>
__device__ __forceinline__ void warp_encode_fast40(const uint32_t* w, uint8_t* sbytes, const uint4* vlut8,
                                                   const uint8_t* scell, __nv_bfloat16* board, size_t row, __nv_bfloat16* glob, int lane) {
    for (int cell = lane; cell < 35; cell += 32) {
        uint64_t bits = cell_bits(w, scell[cell]);
#pragma unroll
        for (int k = 0; k < 5; k++) sbytes[cell * 5 + k] = (uint8_t)(bits >> (8 * k));
    }
    __syncwarp();
    uint32_t pb = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(phase_value(w)));
    uint4* out = reinterpret_cast<uint4*>(board + row * 1400);
    uint8_t* tile = reinterpret_cast<uint8_t*>(board) + (row >> 4) * (size_t)(560 * 128);
    const int leaf = (int)(row & 15);
    for (int v = lane; v < 175; v += 32) {
        uint32_t byte = sbytes[v];
        uint4 o = vlut8[byte];
        if (v % 5 == 4 && (byte & 0x20u)) o.z = (o.z & 0x0000FFFFu) | (pb << 16);   // channel 37 = phase/3
        if (T16K) {
            int cell = v / 5, j = v - 5 * cell, p = cell * 16 + leaf;
            *reinterpret_cast<uint4*>(tile + p * 128 + ((j ^ (p & 7)) << 4)) = o;
        } else {
            out[v] = o;
        }
    }
    for (int g = lane; g < 42; g += 32) glob[g] = __float2bfloat16_rn(global_feature(w, g));
    __syncwarp();
}

// ---- select: move_to_leaf (MCTS.py:63-149) + create_state_tensors(leaf) (MCTS.py:299) ---------
// G = order of the symmetry group of the leaf frames (0: off, the reference's select)
template <typename OT, int LAYOUT, int G>
__global__ void __launch_bounds__(TTPB) k_tree_select(hz_tree T, float cpuct, uint4* leaf_states, OT* board, OT* glob) {
    __shared__ uint32_t sm_words[WPB][32];
    __shared__ uint32_t sm_mask[WPB][40];
    constexpr bool FAST40 = (LAYOUT == HZ_LAYOUT_NHWC40 || LAYOUT == HZ_LAYOUT_T16K) && sizeof(OT) == 2;
    static_assert(LAYOUT != HZ_LAYOUT_T16K || sizeof(OT) == 2, "the T16K image is bf16");
    __shared__ uint4 vlut8[FAST40 ? 256 : 1];
    __shared__ uint8_t sbytes[FAST40 ? WPB : 1][176];
    __shared__ uint8_t scell[36];
    if (FAST40) {
        build_onehot_lut<__nv_bfloat16>(vlut8);
        if (threadIdx.x < 35) scell[threadIdx.x] = CELL_HEX[threadIdx.x];
        __syncthreads();
    }
    int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int t = blockIdx.x * WPB + warp;
    if (t >= active_trees(T)) return;
    TreeView v = view_of(T, t);
    const int K = T.leaves;
    // K descents per tree and step.  K == 1 is the reference's move_to_leaf.  For K > 1 every
    // edge of an already chosen path carries an in-flight visit V: N' = N + V, W' = W - V
    // (a provisional loss for the mover), so the later descents of the step spread out.
    for (int j = 0; j < K; j++) {
        uint32_t* path = v.path + (size_t)j * (T.max_sims + 1);
        int node = 0, depth = 0;
        // (first edge, edge count) of the current node: from the node arrays for the root, afterwards
        // from the winning edge's cached copy, so that a level costs one memory round trip
        uint32_t e0 = v.node_edge0[0];
        int ne = (int)(v.node_info[0] & 0xFFu);
        while (ne != 0) {                                                // is_leaf, MCTS.py:18-20,76
            int N[3]; double W[3]; float P[3]; uint32_t C[3], CI[3];
            int ns = 0;
#pragma unroll
            for (int r = 0; r < 3; r++) {
                int k = lane + 32 * r;
                bool on = k < ne;
                if (32 * r >= ne) { N[r] = 0; W[r] = 0.0; P[r] = 0.0f; C[r] = 0u; CI[r] = 0u; continue; }   // warp-uniform
                if (on) HZ_BOUND(e0 + k, T.max_edges, 101);
                N[r] = on ? v.edge_N[e0 + k] : 0;
                W[r] = on ? v.edge_W[e0 + k] : 0.0;
                P[r] = on ? v.edge_P[e0 + k] : 0.0f;
                C[r] = on ? v.edge_child[e0 + k] : 0u;
                CI[r] = on ? v.edge_cinfo[e0 + k] : 0u;
                if (K > 1 && on) {
                    int vl = v.edge_V[e0 + k];
                    N[r] += vl;
                    W[r] -= (double)vl;
                }
                ns += N[r];
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) ns += __shfl_xor_sync(FULL, ns, o);               // :95-97
            double sqrt_ns = sqrt(ns > 1 ? (double)ns : 1.0);                                  // :99
            double best = -INFINITY;
            int best_k = -1;
#pragma unroll
            for (int r = 0; r < 3; r++) {
                int k = lane + 32 * r;
                if (32 * r >= ne) break;                                 // warp-uniform: most nodes have <= 32 edges
                if (k < ne) {
                    float cp = cpuct * P[r];                             // np.float32 product, :107-109
                    double u = (double)cp * sqrt_ns / (double)(1 + N[r]);                      // :110-111
                    double q = N[r] ? W[r] / (double)N[r] : 0.0;         // Q = W/N, :254
                    double sc = q + u;
                    if (sc > best) { best = sc; best_k = k; }            // strict >, ascending k: :118
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                double ob = __shfl_xor_sync(FULL, best, o);
                int ok = __shfl_xor_sync(FULL, best_k, o);
                bool take = ok >= 0 && (best_k < 0 || ob > best || (ob == best && ok < best_k));
                if (take) { best = ob; best_k = ok; }
            }
            if (best_k < 0) break;                                       // :125-133
            uint32_t e = e0 + (uint32_t)best_k;
            if (depth > T.max_sims) { if (lane == 0) T.status[t] |= 4; break; }
            HZ_BOUND(depth, T.max_sims + 1, 102);
            HZ_BOUND(e, T.max_edges, 103);
            if (lane == 0) {
                path[depth] = e;
                if (K > 1) v.edge_V[e] += 1;
            }
            depth++;
            int br = best_k >> 5;                                        // warp-uniform
            uint32_t wc = br == 0 ? C[0] : br == 1 ? C[1] : C[2], wi = br == 0 ? CI[0] : br == 1 ? CI[1] : CI[2];
            node = (int)__shfl_sync(FULL, wc, best_k & 31);              // :145-146
            HZ_BOUND(node, T.max_nodes, 104);
            uint32_t ci = __shfl_sync(FULL, wi, best_k & 31);
            if (ci == 0) {                                               // not known to be expanded: ask the node
                ne = (int)(v.node_info[node] & 0xFFu);
                if (ne != 0) {
                    e0 = v.node_edge0[node];
                    if (lane == 0) v.edge_cinfo[e] = e0 | ((uint32_t)ne << 24);
                }
            } else {
                e0 = ci & 0xFFFFFFu;
                ne = (int)(ci >> 24);
            }
        }
        if (lane == 0) { T.leaf[t * K + j] = node; T.depth[t * K + j] = depth; }
        size_t row = (size_t)t * K + j;
        warp_load_words(sm_words[warp], v.node_state, node, lane);      // (__syncwarp inside: V updates are visible to the next descent)
        if (leaf_states) reinterpret_cast<uint32_t*>(leaf_states + row * 8)[lane] = sm_words[warp][lane];
        if constexpr (G != 0) {                                          // the network sees T_g(leaf); the tree keeps its frame
            const uint32_t* w = sm_words[warp];
            const int g = sym_frame(w, T.search_key[t], G);
            const uint32_t w22 = w[HZ_W_BAG1META], own = w[lane];
            const uint32_t m = (w22 >> 16) & 0xFFu;
            // the frame is a function of the node within a search: kept in the node's info word, bits 16..27 =
            // g | n_piles << 9 (OR of the same value when the node is reached again; a new search creates new nodes)
            if (lane == 0) atomicOr(&v.node_info[node], ((uint32_t)g | ((m < 5u ? m : 5u) << 9)) << 16);
            if (board) {
                const uint32_t nw = warp_sym_word(own, g, lane);
                __syncwarp();
                sm_words[warp][lane] = nw;
                __syncwarp();
            }
        }
        if (board) {
            if constexpr (FAST40)
                warp_encode_fast40<LAYOUT == HZ_LAYOUT_T16K>(sm_words[warp], sbytes[warp], vlut8, scell, (__nv_bfloat16*)board, row,
                                                             (__nv_bfloat16*)glob + row * 42, lane);
            else
                warp_encode<OT, LAYOUT>(sm_words[warp], sm_mask[warp], board + row * RowElems<LAYOUT>::value, glob + row * 42, lane);
        }
        __syncwarp();
    }
}

// ---- transposition lookup (MCTS.py:184-186) ------------------------------------------------------
// returns node index or -1.  Identity = equality of the 64-bit key, exactly as the reference
// (MCTS.py:185 looks `hash(state)` up in a dict of ids and never compares states); building
// with -DHZ_TREE_FULL_COMPARE=1 additionally compares the 23 key words on a hash match, which
// costs a dependent 128-byte gather per hit and only guards against a 2^-64 collision.
#ifndef HZ_TREE_FULL_COMPARE
#define HZ_TREE_FULL_COMPARE 0
#endif
__device__ __forceinline__ int table_find(const hz_tree& T, const TreeView& v, uint64_t h, const uint32_t* key) {
    uint32_t mask = (uint32_t)T.table_size - 1u;
    uint32_t slot = (uint32_t)h & mask;
    for (uint32_t probes = 0;; probes++) {
        HZ_BOUND(slot, T.table_size, 201);
        HZ_BOUND(probes, T.table_size, 202);      // an open-addressing table of 2x the nodes never fills
        uint32_t e = v.table[slot];
        uint64_t eh = v.table_hash[slot];     // independent of e: both loads are in flight together
        if (e == 0) return -1;
        int idx = (int)e - 1;
        HZ_BOUND(idx, T.max_nodes, 203);
        if (eh == h) {
            if (!HZ_TREE_FULL_COMPARE) return idx;
            State o;
            load_state(o, v.node_state, idx);
            uint32_t ok[HZ_CANON_WORDS];
            key_words(o, T.key_mode, ok);
            bool eq = true;
#pragma unroll
            for (int i = 0; i < HZ_CANON_WORDS; i++) eq &= ok[i] == key[i];
            if (eq) return idx;
        }
        slot = (slot + 1) & mask;
    }
}
__device__ __forceinline__ void table_insert(const hz_tree& T, const TreeView& v, uint64_t h, int idx) {
    uint32_t mask = (uint32_t)T.table_size - 1u;
    uint32_t slot = (uint32_t)h & mask;
    HZ_BOUND(idx, T.max_nodes, 204);
    for (uint32_t probes = 0; atomicCAS(&v.table[slot], 0u, (uint32_t)idx + 1u) != 0u; probes++) {
        HZ_BOUND(probes, T.table_size, 205);
        slot = (slot + 1) & mask;
    }
    v.table_hash[slot] = h;     // read by later rounds only (after the __syncwarp that ends this one)
}

// ---- expand_leaf + terminal value + back_fill (MCTS.py:151-264, 297-352) -------------------------
#ifndef HZ_EXPAND_MIN_BLOCKS
#define HZ_EXPAND_MIN_BLOCKS 4
#endif
// row entry of action a in the evaluator's frame fr (g | n_piles << 9, from the leaf's info word): sigma_g(a)
__device__ __forceinline__ int frame_action(int a, uint32_t fr) {
    const int g = (int)(fr & 0x1FFu), m = (int)(fr >> 9);
    return sym_action(a, g & 3, m, a < m ? sym_pile_perm(g, m, false) : 0u, SYM_HEX_G);
}

// SYM: the leaf rows are in the frames of k_tree_select (hz_tree_set_symmetry); false = the reference's expansion
template <bool SYM>
__global__ void __launch_bounds__(TTPB, HZ_EXPAND_MIN_BLOCKS) k_tree_expand_backup(hz_tree T, const float* policy, const float* value,
                                                             int is_logits, const float* noise, double eps) {
    __shared__ uint32_t sm_words[WPB][32];
    // scoring happens only for children that end the game: read the neighbour LUT in place
    // (global memory, L1-cached) instead of staging 3 KB per block
    const NbrLut* lut = global_nbr_lut();
    int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int t = blockIdx.x * WPB + warp;
    if (t >= active_trees(T)) return;
    TreeView v = view_of(T, t);
    const int K = T.leaves, sim0 = T.sim[t];
    // the K leaves of this step are processed in order j = 0..K-1 (K == 1: the reference)
    for (int j = 0; j < K; j++) {
    const size_t row = (size_t)t * K + j;
    int leaf = T.leaf[row], sim = sim0 + j;
    HZ_BOUND(leaf, T.max_nodes, 306);
    // Everything that depends only on (tree, row, leaf) is requested up front, so that the logits,
    // the tree counters and the statistics of the path edges (back_fill does not depend on the
    // expansion) travel while the leaf state does: the kernel is a chain of dependent round trips.
    const int depth = T.depth[row];
    const uint32_t* path = v.path + (size_t)j * (T.max_sims + 1);
    const float* prow = policy + row * HZ_ACTION_SIZE;
    float pl[5];
    // SYM: the row is loaded through sigma_g (frame in the leaf's info word), so every lane holds what it holds with the mode off
    uint32_t leaf_info = SYM ? v.node_info[leaf] : 0u;
    const uint32_t fr = SYM ? leaf_info >> 16 : 0u;
#pragma unroll
    for (int i = 0; i < 5; i++) {
        const int a = lane + 32 * i;
        pl[i] = a < HZ_ACTION_SIZE ? prow[SYM ? frame_action(a, fr) : a] : -INFINITY;
    }
    const float val_f = value[row];
    const uint32_t pe = lane < depth ? path[lane] : 0u;
    if (!SYM) leaf_info = v.node_info[leaf];
    const uint64_t leaf_hash = v.node_hash[leaf];
    const uint64_t skey = T.search_key[t];
    int n_nodes = T.n_nodes[t];
    const int e0 = T.n_edges[t];
    warp_load_words(sm_words[warp], v.node_state, leaf, lane);
    int p_am = 0, p_N = 0;
    double p_W = 0.0;
    if (lane < depth) { p_am = v.edge_am[pe]; p_N = v.edge_N[pe]; p_W = v.edge_W[pe]; }
    State ls;
    state_from_words(ls, sm_words[warp]);
    int leaf_player = player_of(ls);
    double val;
    if (!is_over(ls)) {                                              // MCTS.py:297
        val = (double)val_f;                                         // :302-304
        // K > 1: a leaf reached twice in one step is expanded by its first simulation only
        bool expand = (leaf_info & 0xFFu) == 0;
        float mx = 0.0f, inv_sum = 1.0f;
        if (is_logits) {                                             // fused softmax (model.py:104)
            float m = fmaxf(fmaxf(fmaxf(pl[0], pl[1]), fmaxf(pl[2], pl[3])), pl[4]);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(FULL, m, o));
            float sum = 0.0f;
#pragma unroll
            for (int i = 0; i < 5; i++) if (lane + 32 * i < HZ_ACTION_SIZE) sum += expf(pl[i] - m);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(FULL, sum, o);
            mx = m; inv_sum = 1.0f / sum;
        }
        Legal L = legal_of(ls);
        int n = expand ? legal_count(L) : 0;
        double noise_sum = 0.0;
        bool mix = noise != nullptr && leaf == 0 && n > 0;           // root Dirichlet, :308-326
        const float* nrow = noise ? noise + (size_t)t * HZ_ACTION_SIZE : nullptr;
        if (mix) {
            uint32_t lw[5];
            legal_words(L, lw);
            for (int a = 0; a < HZ_ACTION_SIZE; a++)                 // sequential fp64 sum, ascending
                if ((lw[a >> 5] >> (a & 31)) & 1u) noise_sum += (double)nrow[a];
        }
        float one_minus = (float)(1.0 - eps);
        int n_new_edges = 0;
        bool overflow = false;
        for (int base = 0; base < n && !overflow; base += 32) {      // expand_leaf, MCTS.py:171-215
            int k = base + lane;
            bool active = k < n;
            int a = active ? kth_action(L, k) : 0;
            State cs = ls;
            uint64_t h = 0;
            uint32_t key[HZ_CANON_WORDS];
            int found = -1;
            if (active) {
                apply_move(cs, a, HZ_NO_DRAW, skey, ((uint32_t)sim << 8) | (uint32_t)a, false, lut);   // :176
                key_words(cs, T.key_mode, key);
                h = hash_key_words(key);                             // :177
                found = table_find(T, v, h, key);                    // :185
            }
            bool selfloop = active && h == leaf_hash;                // :189-194
            // duplicates inside this round (e.g. two identical piles): first lane wins
            bool pending = active && found < 0 && !selfloop;
            unsigned pend_mask = __ballot_sync(FULL, pending);
            int leader = lane;
            if (pending) {
                unsigned same = __match_any_sync(pend_mask, h);
                leader = __ffs(same) - 1;
            }
            // full-key check against the leader (hash equality alone is not identity)
            bool is_dup = pending && leader != lane;
            if (__any_sync(FULL, is_dup)) {
                bool eq = true;
#pragma unroll
                for (int i = 0; i < HZ_CANON_WORDS; i++) {
                    uint32_t lk = __shfl_sync(FULL, key[i], leader);
                    eq &= lk == key[i];
                }
                if (is_dup && !eq) { is_dup = false; leader = lane; }   // 2^-64 event: keep both
            }
            bool is_new = pending && !is_dup;
            unsigned new_mask = __ballot_sync(FULL, is_new);
            int n_new = __popc(new_mask);
            if (n_nodes + n_new > T.max_nodes || e0 + n_new_edges + 32 > T.max_edges) {
                overflow = true;
                if (lane == 0) T.status[t] |= (n_nodes + n_new > T.max_nodes) ? 1 : 2;
                break;
            }
            int id = found;
            if (is_new) {
                id = n_nodes + __popc(new_mask & ((1u << lane) - 1u));
                HZ_BOUND(id, T.max_nodes, 301);
                store_state(cs, v.node_state, id);                   // Node(next_state), :203-204
                v.node_hash[id] = h;
                v.node_edge0[id] = 0;
                v.node_info[id] = (uint32_t)player_of(cs) << 8;
                table_insert(T, v, h, id);
            }
            int leader_id = __shfl_sync(FULL, id, leader);
            if (is_dup) id = leader_id;
            n_nodes += n_new;
            bool valid = active && !selfloop;
            unsigned valid_mask = __ballot_sync(FULL, valid);
            if (valid) {                                             // Edge(...), :212-215
                int e = e0 + n_new_edges + __popc(valid_mask & ((1u << lane) - 1u));
                HZ_BOUND(e, T.max_edges, 302);
                HZ_BOUND(a, HZ_ACTION_SIZE, 303);
                float p = prow[SYM ? frame_action(a, fr) : a];
                if (is_logits) p = expf(p - mx) * inv_sum;
                if (mix) {
                    float keep = one_minus * p;                      // np.float32 product, :323
                    p = (float)((double)keep + eps * ((double)nrow[a] / noise_sum));
                }
                v.edge_child[e] = (uint32_t)id;
                v.edge_N[e] = 0;
                v.edge_V[e] = 0;
                v.edge_cinfo[e] = 0;
                v.edge_W[e] = 0.0;
                v.edge_P[e] = p;
                v.edge_am[e] = (uint16_t)(a | (leaf_player << 8));
            }
            n_new_edges += __popc(valid_mask);
            __syncwarp();
        }
        if (lane == 0 && !overflow && expand) {
            v.node_edge0[leaf] = (uint32_t)e0;
            v.node_info[leaf] = (uint32_t)n_new_edges | ((uint32_t)leaf_player << 8) | (SYM ? (leaf_info & 0xFFFF0000u) : 0u);
            T.n_nodes[t] = n_nodes;
            T.n_edges[t] = e0 + n_new_edges;
        }
    } else {                                                         // terminal leaf, :333-341
        int oc = outcome_of(ls);
        val = oc == 0 ? 0.0 : (leaf_player == 0 ? (double)oc : -(double)oc);
    }
    // back_fill (MCTS.py:220-264): edges of one path are distinct, lanes update them in parallel;
    // the first 32 were fetched at the top
    if (lane < depth) {
        double dir = (p_am >> 8) == leaf_player ? 1.0 : -1.0;        // :242-247
        v.edge_N[pe] = p_N + 1;                                      // :252
        v.edge_W[pe] = p_W + val * dir;                              // :253
        if (K > 1) v.edge_V[pe] -= 1;                                // the in-flight visit has landed
    }
    for (int d = lane + 32; d < depth; d += 32) {
        HZ_BOUND(d, T.max_sims + 1, 304);
        uint32_t e = path[d];
        HZ_BOUND(e, T.max_edges, 305);
        int mover = v.edge_am[e] >> 8;
        double dir = mover == leaf_player ? 1.0 : -1.0;
        v.edge_N[e] += 1;
        v.edge_W[e] += val * dir;
        if (K > 1) v.edge_V[e] -= 1;
    }
    __syncwarp();                                                    // next leaf sees this one's nodes, edges and statistics
    }
    if (lane == 0) T.sim[t] = sim0 + K;
}

// ---- synthetic evaluator (stands in for ModelManager.predict in tests / tree-only benches) -----
// SYM: entry sigma_g(a) of the row gets what entry a gets with the mode off (the frame of k_tree_select)
template <bool SYM>
__global__ void __launch_bounds__(TTPB) k_tree_fake_eval(hz_tree T, float* policy, float* value) {
    __shared__ uint32_t sm_words[WPB][32];
    int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int t = blockIdx.x * WPB + warp;
    if (t >= active_trees(T)) return;
    TreeView v = view_of(T, t);
    for (int j = 0; j < T.leaves; j++) {
        size_t row = (size_t)t * T.leaves + j;
        warp_load_words(sm_words[warp], v.node_state, T.leaf[row], lane);
        State s;
        state_from_words(s, sm_words[warp]);
        uint64_t h = canon_hash(s, HZ_KEY_EXACT);
        const uint32_t fr = SYM ? v.node_info[T.leaf[row]] >> 16 : 0u;
        for (int a = lane; a < HZ_ACTION_SIZE; a += 32)
            policy[row * HZ_ACTION_SIZE + (SYM ? frame_action(a, fr) : a)] = (float)(mix64(h ^ (uint64_t)(a + 1)) >> 40) * 0x1p-24f;
        if (lane == 0) value[row] = (float)((double)(mix64(h ^ 0x5EEDull) >> 40) * 0x1p-23 - 1.0);
        __syncwarp();
    }
}

// ---- rollout evaluator: leaf values from random playouts (hz_tree_rollout_eval) ------------------------------------
// One thread per rollout: thread i*R + r plays rollout r of leaf row i with k_playout's game loop (play_random), shared
// neighbour LUT, rand table and water queue.  With R >= 32 the lanes of a warp start from the same leaf and move in
// lockstep; with R < 32 a warp holds 32/R leaves.  The row's outcomes are summed as integers (shuffles inside the R lanes,
// shared memory across the block's two warps for R = 64), so the value does not depend on the order of the sum.
// 64-thread blocks under (64, 7) for the reason given at k_playout: the register cap leaves the round path room.
constexpr int RTPB = 64;
constexpr int ROLLOUT_MAX_STEPS = 1000;
// SYM: the priors go into the frame of k_tree_select (entry sigma_g(a) gets what entry a gets with the mode off)
template <bool SYM>
__global__ void __launch_bounds__(RTPB, 7) k_tree_rollout_eval(hz_tree T, int log2r, float* policy, float* value,
                                                               unsigned long long* total_steps) {
    const int R = 1 << log2r;
    const int64_t rows = (int64_t)active_trees(T) * T.leaves;
    if ((int64_t)blockIdx.x * RTPB >= (rows << log2r)) return;      // the whole block lies past the active rows
    __shared__ NbrLut lut;
    __shared__ __align__(16) uint64_t rtab_s[RTAB_N];
    __shared__ WaterQueue<2 * RTPB, 2 * RTPB> wq;
    __shared__ int warp_sum[RTPB / 32];
    build_nbr_lut(&lut);
    build_rand_table(rtab_s);
    const RandTab rtab = rand_table_handle(rtab_s);
    water_queue_init(&wq);
    __syncthreads();
    const int64_t gid = (int64_t)blockIdx.x * RTPB + threadIdx.x, row = gid >> log2r;
    const int r = (int)(gid & (R - 1));
    const bool on = row < rows;
    uint32_t k = 0;
    int s0 = 0, s1 = 0, sigma = 0;
    bool fin = false, leaf_over = true;
    State s;
    if (on) {
        const int t = (int)(row / T.leaves), leaf = T.leaf[row];
        HZ_BOUND(leaf, T.max_nodes, 501);
        load_state(s, T.node_state + (size_t)t * T.max_nodes * 8, leaf);   // the row's R threads read one 128 B line
        leaf_over = is_over(s);
        sigma = player_of(s) ? -1 : 1;
        {   // priors: uniform over the legal moves, the R threads of the row split the 143 entries
            const Legal L = legal_of(s);
            const int n = leaf_over ? 0 : legal_count(L);
            uint32_t lw[5];
            legal_words(L, lw);
            const float p = n ? 1.0f / (float)n : 0.0f;
            const uint32_t fr = SYM ? T.node_info[(size_t)t * T.max_nodes + leaf] >> 16 : 0u;
            for (int a = r; a < HZ_ACTION_SIZE; a += R) {
                const int i = a >> 5;   // selects, not lw[i]: a dynamic index would put lw in local memory
                const uint32_t w = i == 0 ? lw[0] : i == 1 ? lw[1] : i == 2 ? lw[2] : i == 3 ? lw[3] : lw[4];
                policy[row * HZ_ACTION_SIZE + (SYM ? frame_action(a, fr) : a)] = ((w >> (a & 31)) & 1u) ? p : 0.0f;
            }
        }
        if (!leaf_over) {
            const uint64_t base = rand64(T.search_key[t] ^ HZ_ROLLOUT_SALT, canon_hash(s, HZ_KEY_EXACT));
            const uint64_t key = rand64(base, (uint64_t)r);
            s.w[HZ_W_KEYLO] = (uint32_t)key;
            s.w[HZ_W_KEYHI] = (uint32_t)(key >> 32);
            k = play_random(s, ROLLOUT_MAX_STEPS, &lut, rtab);
            fin = phase_of(s) == HZ_PHASE_OVER && winner_code(s) == 0;
            if (fin) partial_scores(s, &lut, &wq, s0, s1);
        }
    }
    __syncthreads();
    resolve_water(&lut, &wq);
    __syncthreads();
    if (fin) store_final_scores(s, s0 + wq.extra[threadIdx.x * 2], s1 + wq.extra[threadIdx.x * 2 + 1]);
    int sum = on && !leaf_over ? sigma * outcome_of(s) : 0;      // a stuck or capped rollout is not over: 0
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        if (o < R) sum += __shfl_xor_sync(FULL, sum, o);
    if (R == 64) {                                                // block-uniform
        if ((threadIdx.x & 31) == 0) warp_sum[threadIdx.x >> 5] = sum;
        __syncthreads();
        sum = warp_sum[0] + warp_sum[1];
    }
    if (on && r == 0) value[row] = (float)sum / (float)R;
    if (total_steps) {
        uint32_t steps = k;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) steps += __shfl_xor_sync(FULL, steps, o);
        if ((threadIdx.x & 31) == 0 && steps) atomicAdd(total_steps, (unsigned long long)steps);
    }
}

// ---- frames of the last select (hz_tree_leaf_frames) ------------------------------------------------
__global__ void __launch_bounds__(TTPB) k_tree_leaf_frames(hz_tree T, int on, uint16_t* frames) {
    const int64_t row = (int64_t)blockIdx.x * TTPB + threadIdx.x;
    if (row >= (int64_t)T.n_trees * T.leaves) return;
    const int64_t t = row / T.leaves;
    frames[row] = on ? (uint16_t)((T.node_info[t * T.max_nodes + T.leaf[row]] >> 16) & 0x1FFu) : (uint16_t)0;
}

// ---- root statistics (MCTS.py:355-381) and move choice (MCTS.py:394-441) -------------------------
__global__ void __launch_bounds__(TTPB) k_tree_root_policy(hz_tree T, int32_t* visits, float* pi) {
    int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int t = blockIdx.x * WPB + warp;
    if (t >= T.n_trees) return;
    TreeView v = view_of(T, t);
    int ne = (int)(v.node_info[0] & 0xFFu);
    uint32_t e0 = v.node_edge0[0];
    int total = 0;
    for (int k = lane; k < ne; k += 32) total += v.edge_N[e0 + k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(FULL, total, o);
    for (int a = lane; a < HZ_ACTION_SIZE; a += 32) {
        if (visits) visits[(size_t)t * HZ_ACTION_SIZE + a] = 0;
        if (pi) pi[(size_t)t * HZ_ACTION_SIZE + a] = 0.0f;
    }
    __syncwarp();
    for (int k = lane; k < ne; k += 32) {
        int a = v.edge_am[e0 + k] & 0xFF, N = v.edge_N[e0 + k];
        if (visits) visits[(size_t)t * HZ_ACTION_SIZE + a] = N;
        if (pi && total > 0) pi[(size_t)t * HZ_ACTION_SIZE + a] = (float)((double)N / (double)total);   // :379-381
    }
}

__global__ void __launch_bounds__(TTPB) k_tree_choose(hz_tree T, const float* u01, const uint8_t* exploratory, int16_t* actions) {
    int t = blockIdx.x * TTPB + threadIdx.x;
    if (t >= T.n_trees) return;
    TreeView v = view_of(T, t);
    int ne = (int)(v.node_info[0] & 0xFFu);
    uint32_t e0 = v.node_edge0[0];
    long total = 0;
    for (int k = 0; k < ne; k++) total += v.edge_N[e0 + k];
    int best = -1;
    if (total > 0) {
        bool expl = u01 && (!exploratory || exploratory[t]);
        if (expl) {                                                  // sample ~ N, :404-411
            double thr = (double)u01[t] * (double)total;
            long acc = 0;
            for (int k = 0; k < ne; k++) {
                int N = v.edge_N[e0 + k];
                if (N <= 0) continue;
                acc += N;
                best = v.edge_am[e0 + k] & 0xFF;
                if ((double)acc > thr) break;
            }
        } else {                                                     // first max N, :420-423
            int bestN = 0;
            for (int k = 0; k < ne; k++) {
                int N = v.edge_N[e0 + k];
                if (N > bestN) { bestN = N; best = v.edge_am[e0 + k] & 0xFF; }
            }
        }
    }
    actions[t] = (int16_t)best;
}

__global__ void __launch_bounds__(TTPB) k_tree_root_edges(hz_tree T, int32_t* N, double* W, float* P, int32_t* child) {
    int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int t = blockIdx.x * WPB + warp;
    if (t >= T.n_trees) return;
    TreeView v = view_of(T, t);
    int ne = (int)(v.node_info[0] & 0xFFu);
    uint32_t e0 = v.node_edge0[0];
    size_t row = (size_t)t * HZ_ACTION_SIZE;
    for (int a = lane; a < HZ_ACTION_SIZE; a += 32) {
        if (N) N[row + a] = 0;
        if (W) W[row + a] = 0.0;
        if (P) P[row + a] = 0.0f;
        if (child) child[row + a] = -1;
    }
    __syncwarp();
    for (int k = lane; k < ne; k += 32) {
        int a = v.edge_am[e0 + k] & 0xFF;
        if (N) N[row + a] = v.edge_N[e0 + k];
        if (W) W[row + a] = v.edge_W[e0 + k];
        if (P) P[row + a] = v.edge_P[e0 + k];
        if (child) child[row + a] = (int32_t)v.edge_child[e0 + k];
    }
}

}  // namespace hz

using namespace hz;

// ---- workspace layout ------------------------------------------------------------------------------
static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

struct Layout {
    int max_nodes, max_edges, table_size;
    size_t off[21], total;
};
static Layout layout_for(int n_trees, int max_sims, int max_nodes, int leaves) {
    Layout L;
    L.max_nodes = max_nodes > 0 ? max_nodes : 1 + 69 * max_sims;
    L.max_edges = 69 * max_sims + 32;   // <= 69 edges per expansion, one expansion per simulation
    int ts = 64;
    while (ts < 2 * L.max_nodes) ts <<= 1;
    L.table_size = ts;
    size_t nt = (size_t)n_trees, nn = nt * L.max_nodes, ne = nt * L.max_edges;
    size_t K = (size_t)leaves;
    size_t sizes[21] = {nn * 128, nn * 8, nn * 4, nn * 4, ne * 4, ne * 4, ne * 8, ne * 4, ne * 2,
                        nt * ts * 4, nt * K * (size_t)(max_sims + 1) * 4, nt * K * 4, nt * K * 4, nt * 4, nt * 4, nt * 4, nt, nt * 8,
                        ne * 4, nt * ts * 8, ne * 4};
    size_t o = 0;
    for (int i = 0; i < 21; i++) { L.off[i] = o; o += align256(sizes[i]); }
    L.total = o;
    return L;
}

static inline int tree_blocks(int n, int per_block) { return (n + per_block - 1) / per_block; }

extern "C" {

size_t hz_tree_workspace_bytes(int n_trees, int max_sims, int max_nodes, int leaves) {
    if (n_trees <= 0 || max_sims <= 0 || leaves <= 0 || leaves > 64) return 0;
    return layout_for(n_trees, max_sims, max_nodes, leaves).total;
}

int hz_tree_create(hz_tree** out, void* workspace, size_t workspace_bytes, int n_trees, int max_sims, int max_nodes,
                   int key_mode, int leaves) {
    if (!out || !workspace || n_trees <= 0 || max_sims <= 0 || leaves <= 0 || leaves > 64) return HZ_ERR_ARG;
    if (key_mode != HZ_KEY_EXACT && key_mode != HZ_KEY_REFERENCE) return HZ_ERR_ARG;
    Layout L = layout_for(n_trees, max_sims, max_nodes, leaves);
    if (L.max_edges >= (1 << 24)) return HZ_ERR_ARG;     // edge_cinfo packs the first-edge index into 24 bits
    if (workspace_bytes < L.total || ((uintptr_t)workspace & 255)) return HZ_ERR_WORKSPACE;
    hz_tree* t = new hz_tree;
    char* b = (char*)workspace;
    t->n_trees = n_trees; t->max_sims = max_sims; t->max_nodes = L.max_nodes; t->max_edges = L.max_edges;
    t->table_size = L.table_size; t->key_mode = key_mode; t->leaves = leaves;
    t->node_state = (uint4*)(b + L.off[0]); t->node_hash = (uint64_t*)(b + L.off[1]);
    t->node_edge0 = (uint32_t*)(b + L.off[2]); t->node_info = (uint32_t*)(b + L.off[3]);
    t->edge_child = (uint32_t*)(b + L.off[4]); t->edge_N = (int32_t*)(b + L.off[5]);
    t->edge_W = (double*)(b + L.off[6]); t->edge_P = (float*)(b + L.off[7]); t->edge_am = (uint16_t*)(b + L.off[8]);
    t->table = (uint32_t*)(b + L.off[9]); t->path = (uint32_t*)(b + L.off[10]);
    t->depth = (int32_t*)(b + L.off[11]); t->leaf = (int32_t*)(b + L.off[12]); t->sim = (int32_t*)(b + L.off[13]);
    t->n_nodes = (int32_t*)(b + L.off[14]); t->n_edges = (int32_t*)(b + L.off[15]);
    t->status = (uint8_t*)(b + L.off[16]); t->search_key = (uint64_t*)(b + L.off[17]);
    t->edge_V = (int32_t*)(b + L.off[18]);
    t->table_hash = (uint64_t*)(b + L.off[19]); t->edge_cinfo = (uint32_t*)(b + L.off[20]);
    t->table_bytes = (size_t)n_trees * L.table_size * 4;
    t->n_active = nullptr;
    t->sym_mode = HZ_SYM_OFF;
    t->frames_on = 0;
    *out = t;
    return HZ_OK;
}

int hz_tree_destroy(hz_tree* t) {
    delete t;
    return HZ_OK;
}

int hz_tree_set_active(hz_tree* t, const int32_t* n_active) {
    if (!t || ((uintptr_t)n_active & 3)) return HZ_ERR_ARG;
    t->n_active = n_active;
    return HZ_OK;
}

int hz_tree_set_symmetry(hz_tree* t, int mode) {
    if (!t || (mode != HZ_SYM_OFF && mode != HZ_SYM_BOARD && mode != HZ_SYM_FULL)) return HZ_ERR_ARG;
    t->sym_mode = mode;
    return HZ_OK;
}

int hz_tree_leaf_frames(hz_tree* t, uint16_t* frames, void* stream) {
    if (!t || !frames) return HZ_ERR_ARG;
    k_tree_leaf_frames<<<tree_blocks(t->n_trees * t->leaves, TTPB), TTPB, 0, (cudaStream_t)stream>>>(*t, t->frames_on, frames);
    return hz_launched(1);
}

int hz_tree_reset(hz_tree* t, const void* root_states, const uint64_t* search_keys, void* stream) {
    if (!t || !root_states) return HZ_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(t->table, 0, t->table_bytes, st);
    if (e != cudaSuccess) return hz_record_launch(0, e);
    k_tree_reset<<<tree_blocks(t->n_trees, TTPB), TTPB, 0, st>>>(*t, (const uint4*)root_states, search_keys);
    return hz_launched(1);
}

int hz_tree_select(hz_tree* t, float cpuct, void* leaf_states, void* board, void* glob, int dtype, int layout, void* stream) {
    if (!t || (board && !glob)) return HZ_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    int grid = tree_blocks(t->n_trees, WPB);
    uint4* ls = (uint4*)leaf_states;
    if (layout != HZ_LAYOUT_NCHW && layout != HZ_LAYOUT_NHWC && layout != HZ_LAYOUT_NHWC40 && layout != HZ_LAYOUT_T16K) return HZ_ERR_ARG;
    if (layout == HZ_LAYOUT_T16K && dtype != HZ_DTYPE_BF16) return HZ_ERR_ARG;
#define HZ_SELECT(T, L)                                                                                    \
    (t->sym_mode == HZ_SYM_FULL    ? k_tree_select<T, L, 480><<<grid, TTPB, 0, st>>>(*t, cpuct, ls, (T*)board, (T*)glob) \
     : t->sym_mode == HZ_SYM_BOARD ? k_tree_select<T, L, 4><<<grid, TTPB, 0, st>>>(*t, cpuct, ls, (T*)board, (T*)glob)   \
                                   : k_tree_select<T, L, 0><<<grid, TTPB, 0, st>>>(*t, cpuct, ls, (T*)board, (T*)glob))
    if (dtype == HZ_DTYPE_F32) {
        if (layout == HZ_LAYOUT_NHWC40) HZ_SELECT(float, HZ_LAYOUT_NHWC40);
        else if (layout == HZ_LAYOUT_NHWC) HZ_SELECT(float, HZ_LAYOUT_NHWC);
        else HZ_SELECT(float, HZ_LAYOUT_NCHW);
    } else if (dtype == HZ_DTYPE_BF16) {
        if (layout == HZ_LAYOUT_T16K) HZ_SELECT(__nv_bfloat16, HZ_LAYOUT_T16K);
        else if (layout == HZ_LAYOUT_NHWC40) HZ_SELECT(__nv_bfloat16, HZ_LAYOUT_NHWC40);
        else if (layout == HZ_LAYOUT_NHWC) HZ_SELECT(__nv_bfloat16, HZ_LAYOUT_NHWC);
        else HZ_SELECT(__nv_bfloat16, HZ_LAYOUT_NCHW);
    } else {
        return HZ_ERR_ARG;
    }
#undef HZ_SELECT
    t->frames_on = t->sym_mode != HZ_SYM_OFF;
    return hz_launched(1);
}

int hz_tree_expand_backup(hz_tree* t, const float* policy, const float* value, int is_logits, const float* noise,
                          double eps, void* stream) {
    if (!t || !policy || !value) return HZ_ERR_ARG;
    if (t->sym_mode != HZ_SYM_OFF)
        k_tree_expand_backup<true><<<tree_blocks(t->n_trees, WPB), TTPB, 0, (cudaStream_t)stream>>>(*t, policy, value, is_logits, noise, eps);
    else
        k_tree_expand_backup<false><<<tree_blocks(t->n_trees, WPB), TTPB, 0, (cudaStream_t)stream>>>(*t, policy, value, is_logits, noise, eps);
    return hz_launched(1);
}

int hz_tree_fake_eval(hz_tree* t, float* policy, float* value, void* stream) {
    if (!t || !policy || !value) return HZ_ERR_ARG;
    if (t->sym_mode != HZ_SYM_OFF)
        k_tree_fake_eval<true><<<tree_blocks(t->n_trees, WPB), TTPB, 0, (cudaStream_t)stream>>>(*t, policy, value);
    else
        k_tree_fake_eval<false><<<tree_blocks(t->n_trees, WPB), TTPB, 0, (cudaStream_t)stream>>>(*t, policy, value);
    return hz_launched(1);
}

int hz_tree_rollout_eval(hz_tree* t, int rollouts, float* policy, float* value, unsigned long long* total_steps,
                         void* stream) {
    if (!t || !policy || !value || rollouts < 1 || rollouts > 64 || (rollouts & (rollouts - 1))) return HZ_ERR_ARG;
    int log2r = 0;
    while ((1 << log2r) < rollouts) log2r++;
    int64_t threads = (int64_t)t->n_trees * t->leaves * rollouts;
    const unsigned grid = (unsigned)((threads + RTPB - 1) / RTPB);
    if (t->sym_mode != HZ_SYM_OFF)
        k_tree_rollout_eval<true><<<grid, RTPB, 0, (cudaStream_t)stream>>>(*t, log2r, policy, value, total_steps);
    else
        k_tree_rollout_eval<false><<<grid, RTPB, 0, (cudaStream_t)stream>>>(*t, log2r, policy, value, total_steps);
    return hz_launched(1);
}

int hz_tree_root_policy(hz_tree* t, int32_t* visits, float* pi, void* stream) {
    if (!t || (!visits && !pi)) return HZ_ERR_ARG;
    k_tree_root_policy<<<tree_blocks(t->n_trees, WPB), TTPB, 0, (cudaStream_t)stream>>>(*t, visits, pi);
    return hz_launched(1);
}

int hz_tree_choose(hz_tree* t, const float* u01, const uint8_t* exploratory, int16_t* actions, void* stream) {
    if (!t || !actions) return HZ_ERR_ARG;
    k_tree_choose<<<tree_blocks(t->n_trees, TTPB), TTPB, 0, (cudaStream_t)stream>>>(*t, u01, exploratory, actions);
    return hz_launched(1);
}

int hz_tree_stats(hz_tree* t, int32_t* n_nodes, int32_t* n_edges, uint8_t* status, void* stream) {
    if (!t) return HZ_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaSuccess;
    if (n_nodes) e = cudaMemcpyAsync(n_nodes, t->n_nodes, (size_t)t->n_trees * 4, cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess && n_edges) e = cudaMemcpyAsync(n_edges, t->n_edges, (size_t)t->n_trees * 4, cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess && status) e = cudaMemcpyAsync(status, t->status, (size_t)t->n_trees, cudaMemcpyDeviceToDevice, st);
    return hz_record_launch(0, e);
}

int hz_tree_root_edges(hz_tree* t, int32_t* N, double* W, float* P, int32_t* child, void* stream) {
    if (!t) return HZ_ERR_ARG;
    k_tree_root_edges<<<tree_blocks(t->n_trees, WPB), TTPB, 0, (cudaStream_t)stream>>>(*t, N, W, P, child);
    return hz_launched(1);
}

}  // extern "C"
