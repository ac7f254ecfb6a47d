// hz_evalcache.cuh — the leaf evaluation cache (include/harmonies_b200.h "Leaf evaluation cache"): the handle and the
// device-side probe that k_tree_select<..., CACHE = true> runs on a leaf it has staged in shared memory.
//   entries : set-associative buckets of EC_WAYS ways; entry e holds (exact key, frame) -> the evaluator's row
//             (143 fp32 policy entries + the fp32 value) and a stamp (step of its last insert or hit + 1; 0 = empty)
//   pending : per network row m of the current step, the (key, frame) of its leaf, written by the select and read by
//             hz_evalcache_fill when it inserts the row
#pragma once
#include "hz_core.cuh"

#ifndef HZ_TREE_FULL_COMPARE
#define HZ_TREE_FULL_COMPARE 0
#endif

constexpr int EC_WAYS = 8;
constexpr int EC_ROW = HZ_ACTION_SIZE + 1;      // policy row, then the value
constexpr uint32_t EC_BUSY = 0xFFFFFFFFu;       // stamp of an entry that a fill warp is writing
constexpr int EC_COUNTERS = 6;                  // looked up, hits, terminal, misses, inserts, evictions

struct hz_evalcache {
    int64_t entries, n_buckets;
    int max_rows;
    uint64_t* key;                  // [entries] canon_hash(leaf, HZ_KEY_EXACT)
    uint32_t* frame;                // [entries] evaluation frame g (0 with the symmetry mode off)
    uint32_t* stamp;                // [entries]
    float* row;                     // [entries][EC_ROW]
    uint32_t* words;                // [entries][23] exact key words (HZ_TREE_FULL_COMPARE only)
    uint64_t* pend_key;             // [max_rows]
    uint32_t* pend_frame;           // [max_rows]
    uint32_t* pend_words;           // [max_rows][23] (HZ_TREE_FULL_COMPARE only)
    unsigned long long* counters;   // [EC_COUNTERS]
    uint32_t* clock;                // [0] steps filled so far, [1] block ticket of the running fill
};

// the select's outputs when it runs with a cache
struct EvalCacheArgs {
    hz_evalcache c;
    float* policy;
    float* value;
    int32_t* eval_rows;
    int32_t* n_eval;
};

namespace hz {

// is_over of staged words: the ending flag and a winner
__device__ __forceinline__ bool words_over(const uint32_t* w) {
    const uint32_t m = w[HZ_W_BAG1META];
    return ((m >> 28) & 1u) && ((m >> 29) & 3u);
}

__device__ __forceinline__ int64_t ec_bucket_base(const hz_evalcache& c, uint64_t key) {
    return (int64_t)(((key >> 32) * (uint64_t)c.n_buckets) >> 32) * EC_WAYS;
}

// Warp-cooperative lookup of (key, frame): the entry index, or -1 (every lane gets the answer).  w = the leaf's staged
// words, compared with the entry's key words under HZ_TREE_FULL_COMPARE.
__device__ __forceinline__ int64_t ec_probe(const hz_evalcache& c, uint64_t key, uint32_t fr, const uint32_t* w, int lane) {
    const int64_t base = ec_bucket_base(c, key);
    bool hit = false;
    if (lane < EC_WAYS) {
        const int64_t e = base + lane;
        HZ_BOUND(e, c.entries, 601);
        hit = c.stamp[e] != 0u && c.key[e] == key && c.frame[e] == fr;
        if (HZ_TREE_FULL_COMPARE && hit) {
#pragma unroll
            for (int i = 0; i < HZ_CANON_WORDS; i++)
                hit &= c.words[e * HZ_CANON_WORDS + i] == (i == HZ_W_BAG1META ? (w[i] & 0x0FFFFFFFu) : w[i]);
        }
    }
    const unsigned m = __ballot_sync(0xFFFFFFFFu, hit);
    return m ? base + (__ffs(m) - 1) : -1;
}

}  // namespace hz
