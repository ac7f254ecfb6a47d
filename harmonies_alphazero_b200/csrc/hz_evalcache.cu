// hz_evalcache.cu — the leaf evaluation cache (include/harmonies_b200.h "Leaf evaluation cache"): workspace layout,
// clear / stats, and the fill kernel that scatters the network's compact output back to the tree's leaf rows and inserts
// it.  The lookup runs inside k_tree_select (hz_mcts.cu, hz_tree_select_cached).
#include "hz_common.cuh"
#include "hz_evalcache.cuh"

namespace hz {

constexpr int FPB = 4;   // warps (network rows) per block of the fill

// One warp per network row m < *n_eval: row r = eval_rows[m] of (policy, value) gets the network's row m, and the row is
// inserted into the bucket of its (key, frame).  A way is claimed by a CAS of its stamp to EC_BUSY: the least recently
// stamped way of the bucket (an empty one first); a warp that loses every race drops its insert (a lost hit, never a
// wrong one).  Two rows of one key in a step may both be inserted: their bits are equal.
__global__ void __launch_bounds__(FPB * 32) k_evalcache_fill(hz_evalcache c, const float* net_logits, const float* net_value,
                                                             const int32_t* eval_rows, const int32_t* n_eval, float* policy,
                                                             float* value) {
    __shared__ unsigned long long s_ins, s_evict;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) { s_ins = 0; s_evict = 0; }
    __syncthreads();
    const int n = min(*n_eval, c.max_rows);
    const uint32_t stamp = c.clock[0] + 1u;
    const int m = blockIdx.x * FPB + warp;
    if (m < n) {
        const int r = eval_rows[m];
        HZ_BOUND(r, c.max_rows, 611);
        const uint64_t key = c.pend_key[m];
        const uint32_t fr = c.pend_frame[m];
        long long e = -1;
        uint32_t old = 0;
        if (lane == 0) {
            const int64_t base = ec_bucket_base(c, key);
            for (int tries = 0; tries < EC_WAYS && e < 0; tries++) {
                int best = -1;
                uint32_t bs = EC_BUSY;
                for (int w = 0; w < EC_WAYS; w++) {
                    HZ_BOUND(base + w, c.entries, 612);
                    const uint32_t sw = *(volatile uint32_t*)&c.stamp[base + w];
                    if (sw < bs) { bs = sw; best = w; }
                }
                if (best < 0) break;                                   // every way is being written by another warp
                if (atomicCAS(&c.stamp[base + best], bs, EC_BUSY) == bs) { e = base + best; old = bs; }
            }
        }
        e = __shfl_sync(0xFFFFFFFFu, e, 0);
        const float* src = net_logits + (size_t)m * HZ_ACTION_SIZE;
        for (int a = lane; a < HZ_ACTION_SIZE; a += 32) {
            const float x = src[a];
            policy[(size_t)r * HZ_ACTION_SIZE + a] = x;
            if (e >= 0) c.row[e * EC_ROW + a] = x;
        }
        if (HZ_TREE_FULL_COMPARE && e >= 0 && lane < HZ_CANON_WORDS)
            c.words[e * HZ_CANON_WORDS + lane] = c.pend_words[(size_t)m * HZ_CANON_WORDS + lane];
        if (lane == 0) {
            const float v = net_value[m];
            value[r] = v;
            if (e >= 0) {
                c.row[e * EC_ROW + HZ_ACTION_SIZE] = v;
                c.key[e] = key;
                c.frame[e] = fr;
                __threadfence();                                        // the entry is whole before its stamp is
                c.stamp[e] = stamp;
                atomicAdd(&s_ins, 1ull);
                if (old != 0u) atomicAdd(&s_evict, 1ull);
            }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_ins) atomicAdd(&c.counters[4], s_ins);
        if (s_evict) atomicAdd(&c.counters[5], s_evict);
        if (blockIdx.x == 0 && n > 0) atomicAdd(&c.counters[3], (unsigned long long)n);
        // the last block of the launch advances the step clock (every block has read it by now)
        __threadfence();
        if (atomicAdd(&c.clock[1], 1u) == gridDim.x - 1) {
            c.clock[1] = 0;
            c.clock[0] = stamp;
        }
    }
}

}  // namespace hz

using namespace hz;

static size_t ec_align256(size_t x) { return (x + 255) & ~(size_t)255; }

namespace {
constexpr int EC_PARTS = 10;
struct EcLayout {
    size_t off[EC_PARTS], total;
};
EcLayout ec_layout(int64_t entries, int max_rows) {
    const size_t E = (size_t)entries, R = (size_t)max_rows, W = HZ_TREE_FULL_COMPARE ? HZ_CANON_WORDS : 0;
    const size_t sizes[EC_PARTS] = {E * 8, E * 4, E * 4, E * EC_ROW * 4, R * 8, R * 4, EC_COUNTERS * 8, 2 * 4, E * W * 4, R * W * 4};
    EcLayout L;
    size_t o = 0;
    for (int i = 0; i < EC_PARTS; i++) { L.off[i] = o; o += ec_align256(sizes[i]); }
    L.total = o;
    return L;
}
bool ec_sizes_ok(int64_t entries, int max_rows) {
    return entries >= EC_WAYS && entries % EC_WAYS == 0 && entries <= ((int64_t)1 << 31) && max_rows > 0 && max_rows <= (1 << 26);
}
}  // namespace

extern "C" {

size_t hz_evalcache_bytes(int64_t entries, int max_rows) {
    return ec_sizes_ok(entries, max_rows) ? ec_layout(entries, max_rows).total : 0;
}

int hz_evalcache_create(hz_evalcache** out, void* workspace, size_t bytes, int64_t entries, int max_rows) {
    if (!out || !workspace || !ec_sizes_ok(entries, max_rows)) return HZ_ERR_ARG;
    const EcLayout L = ec_layout(entries, max_rows);
    if (bytes < L.total || ((uintptr_t)workspace & 255)) return HZ_ERR_WORKSPACE;
    char* b = (char*)workspace;
    hz_evalcache* c = new hz_evalcache;
    c->entries = entries;
    c->n_buckets = entries / EC_WAYS;
    c->max_rows = max_rows;
    c->key = (uint64_t*)(b + L.off[0]);
    c->frame = (uint32_t*)(b + L.off[1]);
    c->stamp = (uint32_t*)(b + L.off[2]);
    c->row = (float*)(b + L.off[3]);
    c->pend_key = (uint64_t*)(b + L.off[4]);
    c->pend_frame = (uint32_t*)(b + L.off[5]);
    c->counters = (unsigned long long*)(b + L.off[6]);
    c->clock = (uint32_t*)(b + L.off[7]);
    c->words = HZ_TREE_FULL_COMPARE ? (uint32_t*)(b + L.off[8]) : nullptr;
    c->pend_words = HZ_TREE_FULL_COMPARE ? (uint32_t*)(b + L.off[9]) : nullptr;
    *out = c;
    return HZ_OK;
}

int hz_evalcache_destroy(hz_evalcache* c) {
    delete c;
    return HZ_OK;
}

int hz_evalcache_clear(hz_evalcache* c, void* stream) {
    if (!c) return HZ_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(c->stamp, 0, (size_t)c->entries * 4, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(c->counters, 0, EC_COUNTERS * 8, st);
    return hz_record_launch(0, e);
}

int hz_evalcache_stats(hz_evalcache* c, int64_t* counters, void* stream) {
    if (!c || !counters) return HZ_ERR_ARG;
    return hz_record_launch(0, cudaMemcpyAsync(counters, c->counters, EC_COUNTERS * 8, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
}

int hz_evalcache_fill(hz_evalcache* c, const float* net_logits, const float* net_value, const int32_t* eval_rows,
                      const int32_t* n_eval, float* policy, float* value, void* stream) {
    if (!c || !net_logits || !net_value || !eval_rows || !n_eval || !policy || !value) return HZ_ERR_ARG;
    const unsigned grid = (unsigned)((c->max_rows + FPB - 1) / FPB);
    k_evalcache_fill<<<grid, FPB * 32, 0, (cudaStream_t)stream>>>(*c, net_logits, net_value, eval_rows, n_eval, policy, value);
    return hz_launched(1);
}

}  // extern "C"
