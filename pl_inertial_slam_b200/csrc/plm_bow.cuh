// Bag-of-words loop-candidate scoring: the reference's vendored DBoW2 on the device.
//
//   bow_transform_kernel  TemplatedVocabulary::transform(features, BowVector)
//                         (3rdparty/DBoW2/include/DBoW2/TemplatedVocabulary.h:1045-1101, descent :1196-1238,
//                         FORB::distance src/DBoW2/FORB.cpp:78-100, BowVector::addWeight / addIfNotExist /
//                         normalize src/DBoW2/BowVector.cpp:31-81)
//   bow_score_kernel      L1Scoring::score (src/DBoW2/ScoringObject.cpp:25-69)
// as called from MapHandler::insertKFBowVectorP / L / PL (src/mapHandler.cpp:3116-3237).
//
// Everything that is floating point is evaluated in the reference's ORDER, because fp64 addition is not
// associative and the scores feed comparisons (lookForLoopCandidates, mapHandler.cpp:3239-3299):
//   * a word's value is its weight added once per occurrence (a loop of `count` additions, not count * w);
//   * the L1 norm is one sequential sum over the words in ascending word id (std::map order);
//   * a score is one sequential sum over the common words in ascending word id.
// The parallel parts are the tree descent (one thread per feature; the node table stays L2-resident), the
// per-set sort of (word, leaf) keys in shared memory, the per-word folds, and -- for scoring -- one warp per
// database vector: 128 coalesced entries at a time are tested against a shared-memory bitmap of the query's word
// ids, the rare candidates find the query value through a shared-memory hash table, and the hit lanes' terms are
// then added in lane order, which is word order.
#pragma once
#include "plm_common.cuh"

namespace plm {

constexpr int BOW_THREADS = 256;

struct VocDev {
    const int32_t *child_start; // n_nodes + 1
    const int32_t *child_ids;
    const uint4 *node_desc;     // n_nodes x 32 B
    const double *node_weight;
    const int32_t *node_word;   // >= 0 on leaves
    int n_nodes;
    int weighting;              // DBoW2::WeightingType: 0 TF_IDF, 1 TF, 2 IDF, 3 BINARY
};

// TemplatedVocabulary::transform(feature, id, weight): first child with the smallest distance, down to a leaf.
__device__ __forceinline__ int bow_descend(const VocDev &v, const Desc &q) {
    int node = 0;
    int c0 = __ldg(v.child_start), c1 = __ldg(v.child_start + 1);
    while (c1 > c0) {
        int best = __ldg(v.child_ids + c0);
        int best_d = hamming256(q, load_desc(v.node_desc, best));
        for (int c = c0 + 1; c < c1; ++c) {
            const int id = __ldg(v.child_ids + c);
            const int d = hamming256(q, load_desc(v.node_desc, id));
            if (d < best_d) {
                best_d = d;
                best = id;
            }
        }
        node = best;
        c0 = __ldg(v.child_start + node);
        c1 = __ldg(v.child_start + node + 1);
    }
    return node;
}

struct BowTransformArgs {
    VocDev voc;
    const uint4 *desc;        // n_rows x 32 B
    const int32_t *set_start; // n_sets + 1: features of set s are rows set_start[s] .. set_start[s+1]-1
    int n_sets;
    int cap;                  // power of two >= the largest set (shared-memory sort width)
    uint32_t *bow_ids;        // entries of set s go to slots set_start[s] ..
    double *bow_vals;
    int32_t *bow_len;         // n_sets
};

inline size_t bow_transform_smem(int cap) { return size_t(cap) * (8 + 8 + 4) + 64; }

// The BowVector of ONE descriptor set (rows lo .. lo + n - 1 of desc, n <= cap), by the whole CTA: written to
// out_ids / out_vals [out_lo, out_lo + len); returns len.  cap (a power of two) is the shared-memory sort width; the result does
// not depend on it.  Shared by bow_transform_kernel (many sets) and bow_transform_slots_kernel (the loop-closure
// database: one set per vocabulary, straight into the database's arenas).
__device__ __forceinline__ int bow_transform_set(const VocDev &voc, const uint4 *desc, long long lo, int n, int cap,
                                                 uint32_t *out_ids, double *out_vals, long long out_lo) {
    extern __shared__ __align__(16) unsigned char bow_smem[];
    unsigned long long *keys = reinterpret_cast<unsigned long long *>(bow_smem);    // cap: (word << 32 | leaf), sorted
    double *vals = reinterpret_cast<double *>(bow_smem + size_t(cap) * 8);          // cap: values in word order
    uint32_t *ids = reinterpret_cast<uint32_t *>(bow_smem + size_t(cap) * 16);      // cap
    __shared__ int s_scan[BOW_THREADS];
    __shared__ double s_norm;
    const int tid = threadIdx.x;
    // 1. tree descent, one feature per thread
    for (int f = tid; f < cap; f += BOW_THREADS) {
        unsigned long long key = KEY64_ABSENT;
        if (f < n && voc.n_nodes > 1) {
            const int leaf = bow_descend(voc, load_desc(desc, lo + f));
            if (__ldg(voc.node_weight + leaf) > 0.0) // stopped words are dropped (:1074)
                key = make_key64(static_cast<uint32_t>(__ldg(voc.node_word + leaf)), static_cast<uint32_t>(leaf));
        }
        keys[f] = key;
    }
    __syncthreads();
    // 2. bitonic sort of the keys (ascending word id == std::map order; absent keys sink to the end)
    for (int k = 2; k <= cap; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < cap; i += BOW_THREADS) {
                const int p = i ^ j;
                if (p > i) {
                    const unsigned long long x = keys[i], y = keys[p];
                    const bool up = (i & k) == 0;
                    if ((x > y) == up) {
                        keys[i] = y;
                        keys[p] = x;
                    }
                }
            }
            __syncthreads();
        }
    }
    // 3. one entry per distinct word: every thread owns a contiguous slice of the sorted keys
    const int per = (cap + BOW_THREADS - 1) / BOW_THREADS;
    const int i0 = tid * per, i1 = min(i0 + per, cap);
    int heads = 0;
    for (int i = i0; i < i1; ++i) {
        const unsigned long long k = keys[i];
        if (k != KEY64_ABSENT && (i == 0 || (keys[i - 1] >> 32) != (k >> 32))) ++heads;
    }
    s_scan[tid] = heads;
    __syncthreads();
    for (int off = 1; off < BOW_THREADS; off <<= 1) { // inclusive Hillis-Steele scan of the head counts
        const int v = tid >= off ? s_scan[tid - off] : 0;
        __syncthreads();
        s_scan[tid] += v;
        __syncthreads();
    }
    const int len = s_scan[BOW_THREADS - 1];
    int pos = s_scan[tid] - heads;
    for (int i = i0; i < i1; ++i) {
        const unsigned long long k = keys[i];
        if (k == KEY64_ABSENT || (i > 0 && (keys[i - 1] >> 32) == (k >> 32))) continue;
        const double w = __ldg(voc.node_weight + static_cast<uint32_t>(k));
        double v = w; // insert(id, w)
        if (voc.weighting <= 1) // TF_IDF / TF: addWeight once per further occurrence
            for (int j = i + 1; j < cap && (keys[j] >> 32) == (k >> 32); ++j) v = __dadd_rn(v, w);
        ids[pos] = static_cast<uint32_t>(k >> 32);
        vals[pos] = v;
        ++pos;
    }
    __syncthreads();
    // 4. BowVector::normalize(L1): sequential sum in word order
    if (tid == 0) {
        double norm = 0.0;
        for (int i = 0; i < len; ++i) norm = __dadd_rn(norm, fabs(vals[i]));
        s_norm = norm;
    }
    __syncthreads();
    const double norm = s_norm;
    for (int i = tid; i < len; i += BOW_THREADS) {
        out_ids[out_lo + i] = ids[i];
        out_vals[out_lo + i] = norm > 0.0 ? __ddiv_rn(vals[i], norm) : vals[i];
    }
    __syncthreads();
    return len;
}

// One CTA per descriptor set.
__global__ void __launch_bounds__(BOW_THREADS) bow_transform_kernel(BowTransformArgs a) {
    for (int s = blockIdx.x; s < a.n_sets; s += gridDim.x) {
        const int lo = __ldg(a.set_start + s);
        const int n = min(max(__ldg(a.set_start + s + 1) - lo, 0), a.cap);
        const int len = bow_transform_set(a.voc, a.desc, lo, n, a.cap, a.bow_ids, a.bow_vals, lo);
        if (threadIdx.x == 0) a.bow_len[s] = len;
    }
}

// ---- loop-closure keyframe database (plm_loopdb_*) ----
// Per vocabulary the database keeps an ids / vals arena and, per keyframe slot, the first entry (start) and the entry
// count (len) of the slot's BowVector; one live flag per slot is shared by both vocabularies.
struct LoopVocArgs {
    VocDev voc;
    long long desc_lo;   // first row of the new keyframe's set in the descriptor arena
    int n;               // features in the set
    int cap;             // power of two >= n (this CTA's sort width)
    long long entry_lo;  // first entry reserved for the set in the arena (n entries are reserved)
    uint32_t *ids;       // the vocabulary's arenas and slot tables
    double *vals;
    long long *start;
    int32_t *len;
};

struct LoopTransformArgs {
    LoopVocArgs v[2];    // one per vocabulary the database scores with
    const uint4 *desc;   // the descriptor arena
    uint8_t *live;       // per slot
    int slot;            // the new keyframe's slot
};

// One CTA per vocabulary: the new keyframe's BowVector straight into the arena at its reserved entries, its slot's
// start / len, and its live flag.
__global__ void __launch_bounds__(BOW_THREADS) bow_transform_slots_kernel(LoopTransformArgs a) {
    const LoopVocArgs &v = a.v[blockIdx.x];
    if (threadIdx.x == 0) {
        v.start[a.slot] = v.entry_lo;
        if (blockIdx.x == 0) a.live[a.slot] = 1;
    }
    const int len = bow_transform_set(v.voc, a.desc, v.desc_lo, v.n, v.cap, v.ids, v.vals, v.entry_lo);
    if (threadIdx.x == 0) v.len[a.slot] = len;
}

struct BowScoreArgs {
    const uint32_t *q_ids; // query vectors: entries of query q at q_start[q] .. + q_len[q]
    const double *q_vals;
    const long long *q_start;
    const int32_t *q_len;
    int n_q;
    const uint32_t *db_ids; // database vectors, same layout
    const double *db_vals;
    const long long *db_start;
    const int32_t *db_len;
    int n_db;
    int q_cap;        // >= the longest query (shared-memory staging)
    int table_slots;  // power of two >= 2 * q_cap: open-addressing hash table word id -> position in the query
    int bitmap_words; // 32-bit words of the query-membership bitmap in shared memory (0: none, hash table only)
    double *scores;   // n_q x n_db: scores[q * n_db + j] = score(query q, db j)
};

constexpr int BOW_SCORE_MAX_WARPS = 16;

// query values | hash table | bitmap + its sentinel word | pending-candidate lists of the CTA's warps (32 x int64 each)
inline size_t bow_score_smem(int q_cap, int table_slots, int bitmap_words) {
    return size_t(q_cap) * 8 + size_t(table_slots) * 8 + ((size_t(bitmap_words + 1) * 4 + 7) & ~size_t(7)) +
           size_t(BOW_SCORE_MAX_WARPS) * 32 * 8;
}

__device__ __forceinline__ uint32_t bow_hash(uint32_t id, int slots) { return (id * 2654435761u) & static_cast<uint32_t>(slots - 1); }

// Membership pre-test: bit `id` of the query's word bitmap; ids beyond the bitmap read the all-ones sentinel word that
// follows it ("maybe": the hash table decides).
__device__ __forceinline__ uint32_t bow_maybe(const uint32_t *bitmap, uint32_t bitmap_words, uint32_t id) {
    return (bitmap[min(id >> 5, bitmap_words)] >> (id & 31u)) & 1u;
}

// Position of word `id` in the staged query, or -1.  0xFFFFFFFF marks an empty slot of the table; no word has this id.
__device__ __forceinline__ int bow_find(const uint2 *table, int slots, uint32_t id) {
    if (id == 0xFFFFFFFFu) return -1;
    uint32_t h = bow_hash(id, slots);
    uint2 t = table[h];
    while (t.x != id && t.x != 0xFFFFFFFFu) {
        h = (h + 1) & static_cast<uint32_t>(slots - 1);
        t = table[h];
    }
    return t.x == id ? static_cast<int>(t.y) : -1;
}

// The first n pending candidates of the warp (entry indices, in entry order), all lanes at once: re-read the word id
// (cache hit), look it up in the query's hash table, fetch the database value -- ONE round trip to memory for up to 32
// candidates -- and form the L1 term |vi - wi| - |vi| - |wi| (ScoringObject.cpp:46-52, every operation rounded).  The
// hit terms are then added in lane order == entry order == ascending word id, the reference's summation order.
__device__ __noinline__ double bow_flush(const BowScoreArgs &a, const double *qv, const uint2 *table, const long long *pend, int n,
                                         double score) {
    const int lane = threadIdx.x & 31;
    __syncwarp();
    double term = 0.0;
    bool hit = false;
    if (lane < n) {
        const long long e = pend[lane];
        const int pos = bow_find(table, a.table_slots, __ldg(a.db_ids + e));
        if (pos >= 0) {
            const double vi = qv[pos], wi = __ldg(a.db_vals + e);
            term = __dsub_rn(__dsub_rn(fabs(__dsub_rn(vi, wi)), fabs(vi)), fabs(wi));
            hit = true;
        }
    }
    unsigned lanes = __ballot_sync(0xFFFFFFFFu, hit);
    while (lanes) {
        const int src = __ffs(lanes) - 1;
        score = __dadd_rn(score, __shfl_sync(0xFFFFFFFFu, term, src));
        lanes &= lanes - 1;
    }
    __syncwarp();
    return score;
}

// A chunk (1024 ids) with more than 32 candidates: a database vector that shares most of its words with the query --
// the keyframe's neighbours in the map, or the keyframe itself.  Flushing 32 at a time would cost one memory round
// trip and one 32-step serial sum per flush.  Instead the chunk is re-read (cache hits) with every lane owning 32
// CONSECUTIVE ids, every lane resolves its candidates (eight value loads in flight at a time) into a thread-local array
// of terms, and the running score is handed from lane to lane, each adding its terms in order: the serial chain is one
// DADD per common word and 32 hand-overs.
__device__ __noinline__ double bow_dense_chunk(const BowScoreArgs &a, const double *qv, const uint2 *table, const uint32_t *bitmap,
                                               long long c0, long long ds, long long end, double score) {
    const int lane = threadIdx.x & 31;
    const long long b = c0 + 32 * lane;
    double t[32];
    int cnt = 0;
    for (int k0 = 0; k0 < 32; k0 += 8) {
        int pos[8];
        double w[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const long long e = b + k0 + u;
            pos[u] = -1;
            w[u] = 0.0;
            if (e >= ds && e < end) {
                const uint32_t id = __ldg(a.db_ids + e);
                if (bow_maybe(bitmap, static_cast<uint32_t>(a.bitmap_words), id)) pos[u] = bow_find(table, a.table_slots, id);
                if (pos[u] >= 0) w[u] = __ldg(a.db_vals + e);
            }
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            if (pos[u] >= 0) {
                const double vi = qv[pos[u]];
                t[cnt++] = __dsub_rn(__dsub_rn(fabs(__dsub_rn(vi, w[u])), fabs(vi)), fabs(w[u]));
            }
        }
    }
    unsigned lanes = __ballot_sync(0xFFFFFFFFu, cnt > 0);
    while (lanes) {
        const int src = __ffs(lanes) - 1;
        if (lane == src)
            for (int c = 0; c < cnt; ++c) score = __dadd_rn(score, t[c]);
        score = __shfl_sync(0xFFFFFFFFu, score, src);
        lanes &= lanes - 1;
    }
    return score;
}

// Four nibbles -> four bytes.
__device__ __forceinline__ uint32_t bow_spread4(uint32_t v) {
    v = (v | (v << 8)) & 0x00FF00FFu;
    return (v | (v << 4)) & 0x0F0F0F0Fu;
}

// grid = (CTAs over the database, queries); a warp per database vector.  Two keyframes share only a handful of the
// vocabulary's 10^5 - 10^6 words, so the kernel is a stream over the database word ids: chunks of 1024 ids, eight
// coalesced 16-byte loads per lane, all issued before the first is looked at (one memory round trip per chunk); each id
// is tested against a BITMAP of the query's word ids in shared memory (one LDS) and the outcomes are collected in one
// 32-bit mask per lane (bit 4 i + c: component c of load i).  Entry order is (load, lane, component), so a candidate's
// position among the chunk's candidates comes from one packed warp prefix sum of the eight per-load counts; candidates
// are written at that position into the warp's pending list and resolved together by bow_flush at the end of the
// vector (or when 32 are pending).  A chunk with more than 32 candidates takes bow_dense_chunk.
// Shared-memory layout of a scoring CTA and the staging of query q: its values, the hash table word id -> position and
// the membership bitmap.  The sizes come from the arguments, so CTAs of one launch may score with different vocabularies.
struct BowScoreSmem {
    double *qv;
    uint2 *table;
    uint32_t *bitmap;
    long long *pend_all;
};

__device__ __forceinline__ BowScoreSmem bow_score_stage(const BowScoreArgs &a, int q) {
    extern __shared__ __align__(16) unsigned char bow_smem[];
    BowScoreSmem s;
    s.qv = reinterpret_cast<double *>(bow_smem);
    s.table = reinterpret_cast<uint2 *>(bow_smem + size_t(a.q_cap) * 8);
    s.bitmap = reinterpret_cast<uint32_t *>(s.table + a.table_slots);
    s.pend_all = reinterpret_cast<long long *>(reinterpret_cast<unsigned char *>(s.bitmap) + ((size_t(a.bitmap_words + 1) * 4 + 7) & ~size_t(7)));
    double *qv = s.qv;
    uint2 *table = s.table;
    uint32_t *bitmap = s.bitmap;
    const long long qs = __ldg(a.q_start + q);
    const int qn = min(__ldg(a.q_len + q), a.q_cap);
    for (int i = threadIdx.x; i < a.bitmap_words; i += blockDim.x) bitmap[i] = 0u;
    if (threadIdx.x == 0) bitmap[a.bitmap_words] = 0xFFFFFFFFu;
    for (int i = threadIdx.x; i < a.table_slots; i += blockDim.x) table[i] = make_uint2(0xFFFFFFFFu, 0u);
    __syncthreads();
    const uint32_t bitmap_bits = static_cast<uint32_t>(a.bitmap_words) * 32u;
    for (int i = threadIdx.x; i < qn; i += blockDim.x) {
        const uint32_t id = __ldg(a.q_ids + qs + i);
        qv[i] = __ldg(a.q_vals + qs + i);
        if (id < bitmap_bits) atomicOr(bitmap + (id >> 5), 1u << (id & 31u));
        uint32_t h = bow_hash(id, a.table_slots); // ids of a BowVector are distinct: every insert claims an empty slot
        while (atomicCAS(&table[h].x, 0xFFFFFFFFu, id) != 0xFFFFFFFFu) h = (h + 1) & static_cast<uint32_t>(a.table_slots - 1);
        table[h].y = static_cast<uint32_t>(i);
    }
    __syncthreads();
    return s;
}

// The per-vector loop, by one warp: the L1 sum of the staged query against the database vector at entries
// [ds, end), before the final -score / 2.
__device__ __forceinline__ double bow_score_vector(const BowScoreArgs &a, const BowScoreSmem &s, long long ds, long long end) {
    const double *qv = s.qv;
    const uint2 *table = s.table;
    const uint32_t *bitmap = s.bitmap;
    const int lane = threadIdx.x & 31;
    long long *pend = s.pend_all + 32 * (threadIdx.x >> 5);
    const bool vec = (reinterpret_cast<uintptr_t>(a.db_ids) & 15) == 0;
    const uint32_t bwords = static_cast<uint32_t>(a.bitmap_words);
    double score = 0.0;
    int n_pend = 0; // warp-uniform
    // 16-byte groups start at a multiple of 4 entries; the group holding `ds` may begin up to 3 entries early and
    // the one holding `end - 1` may reach up to 3 entries further -- inside the same 16 aligned bytes as a valid
    // entry, hence mapped; the validity mask drops them
    const long long A = vec ? (ds & ~3LL) : ds;
    for (long long c0 = A; c0 < end; c0 += 1024) {
        const long long e0 = c0 + 4 * lane; // entry of component 0 of this lane's first load; load i is 128 entries on
        uint4 r[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            r[i] = make_uint4(0, 0, 0, 0);
            const long long e = e0 + 128 * i;
            if (e < end) {
                if (vec) {
                    r[i] = __ldg(reinterpret_cast<const uint4 *>(a.db_ids + e));
                } else { // arena not 16-byte aligned: one id at a time
                    r[i].x = __ldg(a.db_ids + e);
                    if (e + 1 < end) r[i].y = __ldg(a.db_ids + e + 1);
                    if (e + 2 < end) r[i].z = __ldg(a.db_ids + e + 2);
                    if (e + 3 < end) r[i].w = __ldg(a.db_ids + e + 3);
                }
            }
        }
        const int left = static_cast<int>(min(end - e0, 4096LL));   // entries from e0 to the end of the vector
        const int skip = static_cast<int>(min(max(ds - e0, 0LL), 4LL)); // > 0 only in the very first load of the vector
        uint32_t mb = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            uint32_t nib = bow_maybe(bitmap, bwords, r[i].x) | (bow_maybe(bitmap, bwords, r[i].y) << 1) |
                           (bow_maybe(bitmap, bwords, r[i].z) << 2) | (bow_maybe(bitmap, bwords, r[i].w) << 3);
            const int n_valid = min(max(left - 128 * i, 0), 4);
            nib &= (1u << n_valid) - 1u;
            if (i == 0) nib &= ~((1u << skip) - 1u);
            mb |= nib << (4 * i);
        }
        if (!__ballot_sync(0xFFFFFFFFu, mb != 0)) continue;
        // per-load candidate counts of this lane, packed one byte each, and their inclusive prefix over the lanes
        uint32_t x = mb - ((mb >> 1) & 0x55555555u);
        x = (x & 0x33333333u) + ((x >> 2) & 0x33333333u); // a popcount per nibble
        const uint32_t own0 = bow_spread4(x & 0xFFFFu), own1 = bow_spread4(x >> 16);
        uint32_t in0 = own0, in1 = own1;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t t0 = __shfl_up_sync(0xFFFFFFFFu, in0, off), t1 = __shfl_up_sync(0xFFFFFFFFu, in1, off);
            if (lane >= off) {
                in0 += t0; // a byte never exceeds 128 (32 lanes x 4)
                in1 += t1;
            }
        }
        const uint32_t tot0 = __shfl_sync(0xFFFFFFFFu, in0, 31), tot1 = __shfl_sync(0xFFFFFFFFu, in1, 31);
        const int sum0 = static_cast<int>(__vsadu4(tot0, 0u)), total = sum0 + static_cast<int>(__vsadu4(tot1, 0u));
        if (total > 32) {
            if (n_pend) score = bow_flush(a, qv, table, pend, n_pend, score);
            n_pend = 0;
            score = bow_dense_chunk(a, qv, table, bitmap, c0, ds, end, score);
            continue;
        }
        if (n_pend + total > 32) {
            score = bow_flush(a, qv, table, pend, n_pend, score);
            n_pend = 0;
        }
        // rank of the first candidate of load i of this lane = candidates of the loads before i (all lanes) +
        // candidates of load i in the lanes below; every byte stays <= 32 here
        const uint32_t rk0 = tot0 * 0x01010100u + (in0 - own0);
        const uint32_t rk1 = tot1 * 0x01010100u + static_cast<uint32_t>(sum0) * 0x01010101u + (in1 - own1);
        uint32_t m = mb;
        while (m) {
            const int k = __ffs(m) - 1, i = k >> 2;
            const uint32_t rk = ((i < 4 ? rk0 : rk1) >> (8 * (i & 3))) & 0xFFu;
            const uint32_t before = __popc((mb >> (4 * i)) & ((1u << (k & 3)) - 1u));
            pend[n_pend + rk + before] = e0 + 128 * i + (k & 3);
            m &= m - 1;
        }
        n_pend += total;
    }
    if (n_pend) score = bow_flush(a, qv, table, pend, n_pend, score);
    return score;
}

__global__ void __launch_bounds__(512) bow_score_kernel(BowScoreArgs a) {
    const int q = blockIdx.y;
    const BowScoreSmem s = bow_score_stage(a, q);
    const int lane = threadIdx.x & 31;
    const int warps = blockDim.x >> 5;
    const int stride = gridDim.x * warps;
    int j = blockIdx.x * warps + (threadIdx.x >> 5);
    long long nx_ds = 0;
    int nx_dn = 0;
    if (j < a.n_db) {
        nx_ds = __ldg(a.db_start + j);
        nx_dn = __ldg(a.db_len + j);
    }
    for (; j < a.n_db; j += stride) {
        const long long ds = nx_ds;
        const long long end = ds + max(nx_dn, 0);
        if (j + stride < a.n_db) {
            nx_ds = __ldg(a.db_start + j + stride);
            nx_dn = __ldg(a.db_len + j + stride);
        }
        const double score = bow_score_vector(a, s, ds, end);
        if (lane == 0) a.scores[static_cast<size_t>(q) * a.n_db + j] = __ddiv_rn(-score, 2.0);
    }
}

// ---- loop-closure keyframe database: the score row of a new keyframe ----
struct LoopScoreArgs {
    BowScoreArgs s[2]; // per vocabulary (blockIdx.y): query = the new slot, database = every slot, scores = its row
    const uint8_t *live;
};

// grid = (CTAs over the slots, vocabularies).  The new keyframe's slot (written by bow_transform_slots_kernel) against
// every live slot, itself included, through the same per-vector loop as bow_score_kernel: same bitmap, hash table and
// summation order, so every score equals plm_bow_score's bit for bit.  Culled slots are skipped and left unwritten.
__global__ void __launch_bounds__(512) bow_score_row_kernel(LoopScoreArgs r) {
    const BowScoreArgs &a = r.s[blockIdx.y];
    const BowScoreSmem s = bow_score_stage(a, 0);
    const int lane = threadIdx.x & 31;
    const int warps = blockDim.x >> 5;
    for (int j = blockIdx.x * warps + (threadIdx.x >> 5); j < a.n_db; j += gridDim.x * warps) {
        if (!__ldg(r.live + j)) continue;
        const long long ds = __ldg(a.db_start + j);
        const double score = bow_score_vector(a, s, ds, ds + max(__ldg(a.db_len + j), 0));
        if (lane == 0) a.scores[j] = __ddiv_rn(-score, 2.0);
    }
}

// insertKFBowVectorPL's blend of the two rows (mapHandler.cpp:3212-3226), every operation rounded on its own (no FMA):
//   s = 0.0 + (sp * n_pt + sl * n_ls) / n_pl;  s = s + (sp * std_pt + sl * std_ls) / std_pl
// with n_pl = n_pt + n_ls and std_pl = std_ls + std_pt.  The leading 0.0 + turns a -0.0 score into +0.0.
__global__ void bow_blend_kernel(const double *__restrict__ sp, const double *__restrict__ sl, int n, double n_pt, double std_pt,
                                 double n_ls, double std_ls, double *__restrict__ out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const double n_pl = __dadd_rn(n_pt, n_ls), std_pl = __dadd_rn(std_ls, std_pt);
    const double p = sp[j], l = sl[j];
    double s = __dadd_rn(0.0, __ddiv_rn(__dadd_rn(__dmul_rn(p, n_pt), __dmul_rn(l, n_ls)), n_pl));
    s = __dadd_rn(s, __ddiv_rn(__dadd_rn(__dmul_rn(p, std_pt), __dmul_rn(l, std_ls)), std_pl));
    out[j] = s;
}

} // namespace plm
