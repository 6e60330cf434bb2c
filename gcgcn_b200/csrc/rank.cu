// Relation evaluation of GCGCN (the DocRED baseline evaluation of config/Config.py:432-561 and its Ign variant,
// config/Config_bert.py:626-650): every (document, i != j, relation r >= 1) candidate is scored with sigmoid, ranked by
// score (descending, stable: equal scores keep insertion order, as Python's list.sort(reverse=True) does), and the
// precision/recall curve over that ranking gives the best F1, its threshold, the AUC and the F1 at a given threshold.
//
//   candidates  logits/labels/intrain [total_pairs, R] -> score f32 + payload (id << 2 | intrain << 1 | correct)
//   sort        stable LSD radix sort of (~bits(score), payload): 4 passes of 8-bit digits, reduce-then-scan
//               (per-tile digit counts -> one digit-major exclusive scan -> stable in-tile ranking and scatter)
//   curve       per-tile flag counts -> exclusive scan -> x, y, f1 (+ Ign) per position, per-tile first argmax and
//               float64 AUC partials -> one-block finish (fixed-order reduction, w, result struct)
//   decode      ranked ids of the first w + 1 candidates -> (doc, row, col, relation, score)
//   merge       two rankings of disjoint candidate sets with global ids -> the ranking of their union (merge path)
//
// Everything is deterministic: integer counts, a stable sort, a merge without atomics and float64 sums in a fixed
// order.
#include "common.cuh"

namespace gcgcn {

constexpr int RK_THREADS = 256;                    // sort and curve tiles: 8 warps x 32 lanes x 16 items
constexpr int RK_IPT = 16;
constexpr int RK_TILE = RK_THREADS * RK_IPT;       // = GCGCN_RANK_TILE
constexpr int RK_WARPS = RK_THREADS / WARP;
constexpr int RK_RADIX = 256;
constexpr int SCAN_THREADS = 1024;                 // device-wide exclusive scan: 1024 threads x 16 values per block
constexpr int SCAN_CHUNK = SCAN_THREADS * 16;
static_assert(RK_TILE == GCGCN_RANK_TILE, "header and kernels disagree on the tile");
static_assert(RK_THREADS == RK_RADIX, "the downsweep gives every thread one digit");
static_assert(RK_IPT == 16, "curve threads own 16 positions (load16)");

__device__ __forceinline__ uint32_t score_key(float s) { return ~__float_as_uint(s); }
__device__ __forceinline__ float key_score(uint32_t k) { return __uint_as_float(~k); }

// ---- candidates --------------------------------------------------------------------------------------------------
// One CTA per pair row (document b, row i): its n pairs x R cells are contiguous in logits.  A candidate's output
// position in this batch is (pair_ptr[b] - node_ptr[b]) (R - 1) + its rank inside document b (every earlier document
// of the batch has n(n-1) off-diagonal pairs).  Its id is that position + base_id, or, with AT, the position inside
// document b + doc_first[b] (the document's first id in a global candidate numbering).
template <bool AT>
__device__ __forceinline__ void rank_candidates_body(const int* __restrict__ node_ptr,
                                                     const long long* __restrict__ pair_ptr,
                                                     const int* __restrict__ row_doc, const float* __restrict__ z,
                                                     const float* __restrict__ labels,
                                                     const uint8_t* __restrict__ intrain, int R, long long base_id,
                                                     const long long* __restrict__ doc_first, float* __restrict__ score,
                                                     uint32_t* __restrict__ payload,
                                                     unsigned long long* __restrict__ counters) {
    __shared__ unsigned int red[2][8];
    const int row = blockIdx.x;
    const int b = row_doc[row];
    const int n = node_ptr[b + 1] - node_ptr[b], i = row - node_ptr[b];
    const long long cell0 = (pair_ptr[b] + static_cast<long long>(i) * n) * R;
    const long long doc_base = base_id + (pair_ptr[b] - node_ptr[b]) * (R - 1);
    const long long row_base = doc_base + static_cast<long long>(i) * (n - 1) * (R - 1);
    // AT: positions and ids are below 2^30, so 32 bits hold both (no more registers live across the loop than without)
    const uint32_t row_pos = static_cast<uint32_t>(row_base);
    const uint32_t row_id = AT ? static_cast<uint32_t>(doc_first[b] + static_cast<long long>(i) * (n - 1) * (R - 1)) : 0u;
    const int cells = n * R;
    unsigned int pos = 0, nan = 0;
    for (int c = threadIdx.x; c < cells; c += blockDim.x) {
        const int j = c / R, r = c - j * R;
        if (j == i || r == 0) continue;
        const float s = logit_sigmoid(z[cell0 + c]);
        const uint32_t corr = (labels != nullptr && labels[cell0 + c] > 0.5f) ? 1u : 0u;
        const uint32_t intr = (intrain != nullptr && intrain[cell0 + c] != 0) ? 2u : 0u;
        if constexpr (AT) {
            const uint32_t off = static_cast<uint32_t>((j - (j > i)) * (R - 1) + (r - 1));
            score[row_pos + off] = s;
            payload[row_pos + off] = ((row_id + off) << 2) | intr | corr;
        } else {
            const long long id = row_base + static_cast<long long>(j - (j > i)) * (R - 1) + (r - 1);
            score[id - base_id] = s;
            payload[id - base_id] = (static_cast<uint32_t>(id) << 2) | intr | corr;
        }
        pos += corr;
        nan += (s != s) ? 1u : 0u;
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        pos += __shfl_xor_sync(0xffffffffu, pos, o);
        nan += __shfl_xor_sync(0xffffffffu, nan, o);
    }
    if (lane == 0) { red[0][warp] = pos; red[1][warp] = nan; }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int p = 0, q = 0;
        for (int w = 0; w < 8; ++w) { p += red[0][w]; q += red[1][w]; }
        if (p) atomicAdd(counters, static_cast<unsigned long long>(p));
        if (q) atomicAdd(counters + 1, static_cast<unsigned long long>(q));
    }
}

__global__ void __launch_bounds__(256)
rank_candidates_kernel(const int* __restrict__ node_ptr, const long long* __restrict__ pair_ptr,
                       const int* __restrict__ row_doc, const float* __restrict__ z, const float* __restrict__ labels,
                       const uint8_t* __restrict__ intrain, int R, long long base_id, float* __restrict__ score,
                       uint32_t* __restrict__ payload, unsigned long long* __restrict__ counters) {
    rank_candidates_body<false>(node_ptr, pair_ptr, row_doc, z, labels, intrain, R, base_id, nullptr, score, payload,
                                counters);
}

__global__ void __launch_bounds__(256)
rank_candidates_at_kernel(const int* __restrict__ node_ptr, const long long* __restrict__ pair_ptr,
                          const int* __restrict__ row_doc, const float* __restrict__ z,
                          const float* __restrict__ labels, const uint8_t* __restrict__ intrain, int R,
                          const long long* __restrict__ doc_first, float* __restrict__ score,
                          uint32_t* __restrict__ payload, unsigned long long* __restrict__ counters) {
    rank_candidates_body<true>(node_ptr, pair_ptr, row_doc, z, labels, intrain, R, 0LL, doc_first, score, payload,
                               counters);
}

// ---- block-wide exclusive scan of one value per thread (blockDim.x = NT) -----------------------------------------
template <typename T, int NT>
__device__ __forceinline__ T block_excl_scan(T v, T* s_warp, T* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    T inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        T w = lane < NT / 32 ? s_warp[lane] : T(0);
        T wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const T t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += t;
        }
        if (lane < NT / 32) s_warp[lane] = wi - w;
        if (lane == NT / 32 - 1) s_warp[32] = wi;
    }
    __syncthreads();
    const T out = s_warp[warp] + inc - v;
    if (total != nullptr) *total = s_warp[32];
    __syncthreads();
    return out;
}

// v[k] = x[base + k] for the 16 values a thread owns (0 past n): 16-byte loads when all 16 exist (base is a multiple of
// 16 values and x is 256-byte aligned), so a warp's load touches 16-byte pieces instead of one word per lane
template <typename T>
__device__ __forceinline__ void load16(const T* __restrict__ x, long long base, long long n, T (&v)[16]) {
    if (base + 16 <= n) {
        const uint4* x4 = reinterpret_cast<const uint4*>(x + base);
#pragma unroll
        for (int q = 0; q < 16 * static_cast<int>(sizeof(T)) / 16; ++q) reinterpret_cast<uint4*>(v)[q] = x4[q];
    } else {
#pragma unroll
        for (int k = 0; k < 16; ++k) v[k] = base + k < n ? x[base + k] : T(0);
    }
}

// ---- device-wide exclusive scan in place (the sort's digit-major tile counts, the curve's packed flag counts) ------
template <typename T>
__global__ void __launch_bounds__(SCAN_THREADS)
scan_reduce_kernel(const T* __restrict__ x, long long n, T* __restrict__ block_sums) {
    __shared__ T s_warp[33];
    const long long base = static_cast<long long>(blockIdx.x) * SCAN_CHUNK + threadIdx.x * 16LL;
    T v[16];
    load16(x, base, n, v);
    T acc = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) acc += v[k];
    T total;
    block_excl_scan<T, SCAN_THREADS>(acc, s_warp, &total);
    if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

template <typename T>
__global__ void __launch_bounds__(SCAN_THREADS)
scan_top_kernel(T* __restrict__ sums, int n) {
    __shared__ T s_warp[33];
    T carry = 0;
    for (int c0 = 0; c0 < n; c0 += SCAN_THREADS) {
        const int idx = c0 + threadIdx.x;
        const T v = idx < n ? sums[idx] : T(0);
        T total;
        const T ex = block_excl_scan<T, SCAN_THREADS>(v, s_warp, &total);
        if (idx < n) sums[idx] = carry + ex;
        carry += total;
    }
}

template <typename T>
__global__ void __launch_bounds__(SCAN_THREADS)
scan_down_kernel(T* __restrict__ x, long long n, const T* __restrict__ block_sums) {
    __shared__ T s_warp[33];
    const long long base = static_cast<long long>(blockIdx.x) * SCAN_CHUNK + threadIdx.x * 16LL;
    T v[16];
    load16(x, base, n, v);
    T acc = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) acc += v[k];
    T run = block_excl_scan<T, SCAN_THREADS>(acc, s_warp, nullptr) + block_sums[blockIdx.x];
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        if (base + k < n) x[base + k] = run;
        run += v[k];
    }
}

template <typename T>
static int launch_scan(T* x, long long n, T* block_sums, cudaStream_t st) {
    const int blocks = ceil_div(n, SCAN_CHUNK);
    scan_reduce_kernel<T><<<blocks, SCAN_THREADS, 0, st>>>(x, n, block_sums);
    GCGCN_CHECK_LAUNCH("rank_scan_reduce");
    scan_top_kernel<T><<<1, SCAN_THREADS, 0, st>>>(block_sums, blocks);
    GCGCN_CHECK_LAUNCH("rank_scan_top");
    scan_down_kernel<T><<<blocks, SCAN_THREADS, 0, st>>>(x, n, block_sums);
    GCGCN_CHECK_LAUNCH("rank_scan_down");
    return GCGCN_OK;
}

// ---- radix sort -------------------------------------------------------------------------------------------------
// Pass 0 reads the float scores and forms the keys ~bits(s) (scores are >= 0, so the bit pattern is monotone and its
// complement ascends as the score descends); later passes read the keys of the previous pass.
template <bool FIRST>
__device__ __forceinline__ uint32_t load_key(const void* in, long long idx) {
    if (FIRST) return score_key(reinterpret_cast<const float*>(in)[idx]);
    return reinterpret_cast<const uint32_t*>(in)[idx];
}

// Where a pass takes its 8-bit digit: the key formed from the score (the sort's pass 0), the key of the previous pass
// (digit at bit `arg`), or the candidate's relation from the payload, (id mod (R - 1)) with arg = R - 1 (the stable
// partition of a ranking by relation, gcgcn_rank_by_relation).
enum DigitSrc { DIGIT_SCORE, DIGIT_KEY, DIGIT_RELATION };

template <int SRC>
__device__ __forceinline__ uint32_t radix_digit(uint32_t key, uint32_t pay, int arg) {
    if (SRC == DIGIT_RELATION) return (pay >> 2) % static_cast<uint32_t>(arg);
    return (key >> arg) & 255u;
}

// counts[d * tiles + tile] = number of items of the tile whose digit is d; keys_in holds the payloads for
// DIGIT_RELATION
template <int SRC>
__global__ void __launch_bounds__(RK_THREADS)
radix_upsweep_kernel(const void* __restrict__ keys_in, long long count, int shift, int tiles,
                     uint32_t* __restrict__ counts) {
    __shared__ uint32_t hist[RK_WARPS][RK_RADIX];
    const int warp = threadIdx.x >> 5;
    for (int t = threadIdx.x; t < RK_WARPS * RK_RADIX; t += RK_THREADS) (&hist[0][0])[t] = 0u;
    __syncthreads();
    const long long base = static_cast<long long>(blockIdx.x) * RK_TILE;
#pragma unroll 4
    for (int k = 0; k < RK_IPT; ++k) {
        const long long idx = base + k * RK_THREADS + threadIdx.x;
        if (idx < count) {
            const uint32_t x = load_key<SRC == DIGIT_SCORE>(keys_in, idx);
            atomicAdd(&hist[warp][radix_digit<SRC>(x, x, shift)], 1u);
        }
    }
    __syncthreads();
    uint32_t s = 0;
#pragma unroll
    for (int w = 0; w < RK_WARPS; ++w) s += hist[w][threadIdx.x];
    counts[static_cast<long long>(threadIdx.x) * tiles + blockIdx.x] = s;
}

// Stable scatter of one tile.  Warp w owns the tile's items [512 w, 512 w + 512), visited in 16 rounds of 32 in input
// order; in each round the lanes holding the same digit find each other with match.any and take consecutive ranks
// after the warp's running count of that digit.  Tile rank = start of the digit in the tile + the counts of that
// digit in earlier warps + the warp rank.  The tile is staged in shared memory in digit order, then written out so
// that each digit's run is contiguous at offsets[d * tiles + tile] (the digit-major exclusive scan of the counts).
template <int SRC>
__global__ void __launch_bounds__(RK_THREADS)
radix_downsweep_kernel(const void* __restrict__ keys_in, const uint32_t* __restrict__ vals_in, long long count, int shift,
                       int tiles, const uint32_t* __restrict__ offsets, uint32_t* __restrict__ keys_out,
                       uint32_t* __restrict__ vals_out) {
    __shared__ uint32_t s_keys[RK_TILE];
    __shared__ uint32_t s_vals[RK_TILE];
    __shared__ uint32_t s_whist[RK_WARPS][RK_RADIX];
    __shared__ uint32_t s_start[RK_RADIX];
    __shared__ uint32_t s_gout[RK_RADIX];
    __shared__ uint32_t s_warp[33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long base = static_cast<long long>(blockIdx.x) * RK_TILE;
    const int valid = static_cast<int>(min(static_cast<long long>(RK_TILE), count - base));
    for (int t = threadIdx.x; t < RK_WARPS * RK_RADIX; t += RK_THREADS) (&s_whist[0][0])[t] = 0u;
    __syncthreads();

    const uint32_t lt_mask = (1u << lane) - 1u;
    uint32_t key[RK_IPT], val[RK_IPT];
    uint32_t rank[RK_IPT];
#pragma unroll
    for (int k = 0; k < RK_IPT; ++k) {
        const int t = warp * (RK_IPT * WARP) + k * WARP + lane;
        const bool ok = t < valid;
        key[k] = ok ? load_key<SRC == DIGIT_SCORE>(keys_in, base + t) : 0u;
        val[k] = ok ? vals_in[base + t] : 0u;
        const uint32_t d = ok ? radix_digit<SRC>(key[k], val[k], shift) : 256u;
        const uint32_t peers = __match_any_sync(0xffffffffu, d);
        const uint32_t before = ok ? s_whist[warp][d] : 0u;
        __syncwarp();
        if (ok && (peers & lt_mask) == 0u) s_whist[warp][d] = before + __popc(peers);
        __syncwarp();
        rank[k] = before + __popc(peers & lt_mask);
    }
    __syncthreads();
    // thread d: counts of digit d in earlier warps, the digit's start in the tile, its global offset
    {
        const int d = threadIdx.x;
        uint32_t run = 0;
#pragma unroll
        for (int w = 0; w < RK_WARPS; ++w) {
            const uint32_t c = s_whist[w][d];
            s_whist[w][d] = run;
            run += c;
        }
        const uint32_t start = block_excl_scan<uint32_t, RK_THREADS>(run, s_warp, nullptr);
        s_start[d] = start;
        s_gout[d] = offsets[static_cast<long long>(d) * tiles + blockIdx.x];
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < RK_IPT; ++k) {
        const int t = warp * (RK_IPT * WARP) + k * WARP + lane;
        if (t < valid) {
            const uint32_t d = radix_digit<SRC>(key[k], val[k], shift);
            const uint32_t p = s_start[d] + s_whist[warp][d] + rank[k];
            s_keys[p] = key[k];
            s_vals[p] = val[k];
        }
    }
    __syncthreads();
    for (int t = threadIdx.x; t < valid; t += RK_THREADS) {
        const uint32_t k = s_keys[t];
        const uint32_t d = radix_digit<SRC>(k, SRC == DIGIT_RELATION ? s_vals[t] : 0u, shift);
        const long long o = static_cast<long long>(s_gout[d]) + (t - static_cast<int>(s_start[d]));
        keys_out[o] = k;
        vals_out[o] = s_vals[t];
    }
}

struct SortWs {
    uint32_t *keys, *vals, *counts, *sums;
};
static int rank_tiles(long long count) { return ceil_div(count, RK_TILE); }

static bool sort_ws_take(Arena& a, long long count, SortWs* w) {
    const long long tiles = rank_tiles(count);
    const long long counts = tiles * RK_RADIX;
    w->keys = a.take<uint32_t>(count);
    w->vals = a.take<uint32_t>(count);
    w->counts = a.take<uint32_t>(counts);
    w->sums = a.take<uint32_t>(ceil_div(counts, SCAN_CHUNK));
    return w->keys && w->vals && w->counts && w->sums;
}

// curve workspace: per tile the packed flag count (correct | (correct & intrain) << 32) and its scan, the tile's
// first argmax of f1 (value, position), the max of the Ign f1 and the two float64 AUC partials
struct CurveWs {
    unsigned long long *flags, *sums;
    float *best_f1, *best_ign;
    long long* best_pos;
    double *auc, *ign_auc;
};
static bool curve_ws_take(Arena& a, long long count, CurveWs* w) {
    const long long tiles = rank_tiles(count);
    w->flags = a.take<unsigned long long>(tiles);
    w->sums = a.take<unsigned long long>(ceil_div(tiles, SCAN_CHUNK));
    w->best_f1 = a.take<float>(tiles);
    w->best_ign = a.take<float>(tiles);
    w->best_pos = a.take<long long>(tiles);
    w->auc = a.take<double>(tiles);
    w->ign_auc = a.take<double>(tiles);
    return w->flags && w->sums && w->best_f1 && w->best_ign && w->best_pos && w->auc && w->ign_auc;
}

// The scans and the curve read their workspace arrays with 16-byte loads: the arena starts at the first 256-byte
// boundary of the caller's workspace, whatever its alignment (rank_ws_bytes includes the slack).
static Arena rank_arena(void* ws, size_t ws_bytes) {
    const uintptr_t p = reinterpret_cast<uintptr_t>(ws);
    const size_t skip = ((p + 255) & ~uintptr_t(255)) - p;
    if (ws == nullptr || ws_bytes < skip) return Arena(nullptr, 0);
    return Arena(static_cast<char*>(ws) + skip, ws_bytes - skip);
}

size_t rank_ws_bytes(long long count) {
    if (count <= 0) return 512;
    Arena probe(reinterpret_cast<void*>(256), ~size_t(0) >> 1);
    SortWs s;
    sort_ws_take(probe, count, &s);
    const size_t sort_bytes = probe.off;
    Arena probe2(reinterpret_cast<void*>(256), ~size_t(0) >> 1);
    CurveWs c;
    curve_ws_take(probe2, count, &c);
    return std::max(sort_bytes, probe2.off) + 256;
}

int launch_rank_candidates(const gcgcn_batch* bt, const float* z, const float* labels, const uint8_t* intrain, int R,
                           long long base_id, float* score, uint32_t* payload, unsigned long long* counters,
                           cudaStream_t st) {
    if (bt->total_nodes <= 0) return GCGCN_OK;
    rank_candidates_kernel<<<bt->total_nodes, 256, 0, st>>>(bt->node_ptr, reinterpret_cast<const long long*>(bt->pair_ptr),
                                                            bt->row_doc, z, labels, intrain, R, base_id, score, payload,
                                                            counters);
    GCGCN_CHECK_LAUNCH("rank_candidates");
    return GCGCN_OK;
}

int launch_rank_candidates_at(const gcgcn_batch* bt, const float* z, const float* labels, const uint8_t* intrain,
                              int R, const long long* doc_first, float* score, uint32_t* payload,
                              unsigned long long* counters, cudaStream_t st) {
    if (bt->total_nodes <= 0) return GCGCN_OK;
    rank_candidates_at_kernel<<<bt->total_nodes, 256, 0, st>>>(bt->node_ptr,
                                                               reinterpret_cast<const long long*>(bt->pair_ptr),
                                                               bt->row_doc, z, labels, intrain, R, doc_first, score,
                                                               payload, counters);
    GCGCN_CHECK_LAUNCH("rank_candidates_at");
    return GCGCN_OK;
}

int launch_rank_sort(const float* score, const uint32_t* payload, long long count, uint32_t* sorted_key,
                     uint32_t* sorted_payload, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (count <= 0) return GCGCN_OK;
    Arena a = rank_arena(ws, ws_bytes);
    SortWs w;
    if (!sort_ws_take(a, count, &w)) return fail(GCGCN_ERR_WORKSPACE, "rank_sort: workspace too small (%zu bytes)", ws_bytes);
    const int tiles = rank_tiles(count);
    const long long ncounts = static_cast<long long>(tiles) * RK_RADIX;
    // passes: scores -> ws -> out -> ws -> out
    const void* kin = score;
    const uint32_t* vin = payload;
    for (int pass = 0; pass < 4; ++pass) {
        uint32_t* kout = (pass & 1) ? sorted_key : w.keys;
        uint32_t* vout = (pass & 1) ? sorted_payload : w.vals;
        const int shift = 8 * pass;
        if (pass == 0) radix_upsweep_kernel<DIGIT_SCORE><<<tiles, RK_THREADS, 0, st>>>(kin, count, shift, tiles, w.counts);
        else radix_upsweep_kernel<DIGIT_KEY><<<tiles, RK_THREADS, 0, st>>>(kin, count, shift, tiles, w.counts);
        GCGCN_CHECK_LAUNCH("rank_radix_upsweep");
        GCGCN_TRY(launch_scan<uint32_t>(w.counts, ncounts, w.sums, st));
        if (pass == 0)
            radix_downsweep_kernel<DIGIT_SCORE><<<tiles, RK_THREADS, 0, st>>>(kin, vin, count, shift, tiles, w.counts,
                                                                             kout, vout);
        else
            radix_downsweep_kernel<DIGIT_KEY><<<tiles, RK_THREADS, 0, st>>>(kin, vin, count, shift, tiles, w.counts, kout,
                                                                           vout);
        GCGCN_CHECK_LAUNCH("rank_radix_downsweep");
        kin = kout;
        vin = vout;
    }
    return GCGCN_OK;
}

// ---- merge of two sorted runs ------------------------------------------------------------------------------------
// Runs A and B ascend by (key, payload) read as one 64-bit value (key in the high word).  Merge path: output tile t
// holds outputs [t TILE, (t + 1) TILE); the partition kernel finds, for every tile boundary d, how many of the first d
// outputs come from A (a binary search along the diagonal a + b = d).  One CTA per tile stages its A and B slices in
// shared memory, each thread finds its own 16-output diagonal in them and merges 16 outputs, and the tile is written
// back through shared memory as 16-byte stores.  On equal values A comes first.
__device__ __forceinline__ unsigned long long merge_value(uint32_t key, uint32_t pay) {
    return (static_cast<unsigned long long>(key) << 32) | pay;
}

// split[t] = number of A items among the first min(t TILE, na + nb) outputs, t = 0 .. tiles
__global__ void __launch_bounds__(256)
merge_partition_kernel(const uint32_t* __restrict__ key_a, const uint32_t* __restrict__ pay_a, long long na,
                       const uint32_t* __restrict__ key_b, const uint32_t* __restrict__ pay_b, long long nb, int tiles,
                       long long* __restrict__ split) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > tiles) return;
    const long long d = min(static_cast<long long>(t) * RK_TILE, na + nb);
    long long lo = max(0LL, d - nb), hi = min(d, na);
    while (lo < hi) {                      // first i whose A[i] comes after B[d - 1 - i]
        const long long mid = (lo + hi) >> 1;
        const long long j = d - 1 - mid;
        if (merge_value(key_a[mid], pay_a[mid]) <= merge_value(key_b[j], pay_b[j])) lo = mid + 1;
        else hi = mid;
    }
    split[t] = lo;
}

constexpr int MG_PAD = RK_TILE + RK_TILE / WARP;   // output staging: one padding word per 32 (conflict-free)
__device__ __forceinline__ int merge_slot(int p) { return p + (p >> 5); }

__global__ void __launch_bounds__(RK_THREADS)
merge_tile_kernel(const uint32_t* __restrict__ key_a, const uint32_t* __restrict__ pay_a, long long na,
                  const uint32_t* __restrict__ key_b, const uint32_t* __restrict__ pay_b, long long nb,
                  const long long* __restrict__ split, uint32_t* __restrict__ key_out, uint32_t* __restrict__ pay_out) {
    // input staging: A slice then B slice in [0, n) of s_key / s_pay; output staging reuses the same words
    __shared__ __align__(16) uint32_t smem[2 * MG_PAD];
    uint32_t* s_key = smem;
    uint32_t* s_pay = smem + RK_TILE;
    const long long o0 = static_cast<long long>(blockIdx.x) * RK_TILE;
    const long long a0 = split[blockIdx.x], a1 = split[blockIdx.x + 1];
    const long long b0 = o0 - a0;
    const int n = static_cast<int>(min(static_cast<long long>(RK_TILE), na + nb - o0));
    const int nA = static_cast<int>(a1 - a0), nB = n - nA;
    for (int q = threadIdx.x; q < n; q += RK_THREADS) {
        const bool fa = q < nA;
        s_key[q] = fa ? key_a[a0 + q] : key_b[b0 + q - nA];
        s_pay[q] = fa ? pay_a[a0 + q] : pay_b[b0 + q - nA];
    }
    __syncthreads();
    // this thread's outputs [d, d + 16) of the tile start at A index i, B index d - i
    const int d = min(static_cast<int>(threadIdx.x) * RK_IPT, n);
    int lo = max(0, d - nB), hi = min(d, nA);
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const int j = nA + d - 1 - mid;
        if (merge_value(s_key[mid], s_pay[mid]) <= merge_value(s_key[j], s_pay[j])) lo = mid + 1;
        else hi = mid;
    }
    int i = lo, j = nA + d - lo;                   // j indexes the B slice at its staged position
    uint32_t ka = i < nA ? s_key[i] : 0u, pa = i < nA ? s_pay[i] : 0u;
    uint32_t kb = j < n ? s_key[j] : 0u, pb = j < n ? s_pay[j] : 0u;
    uint32_t ok[RK_IPT], op[RK_IPT];
#pragma unroll
    for (int k = 0; k < RK_IPT; ++k) {
        const bool take_a = i < nA && (j >= n || merge_value(ka, pa) <= merge_value(kb, pb));
        ok[k] = take_a ? ka : kb;
        op[k] = take_a ? pa : pb;
        if (take_a) {
            ++i;
            if (i < nA) { ka = s_key[i]; pa = s_pay[i]; }
        } else {
            ++j;
            if (j < n) { kb = s_key[j]; pb = s_pay[j]; }
        }
    }
    __syncthreads();
    uint32_t* o_key = smem;
    uint32_t* o_pay = smem + MG_PAD;
#pragma unroll
    for (int k = 0; k < RK_IPT; ++k) {
        if (d + k < n) {
            o_key[merge_slot(d + k)] = ok[k];
            o_pay[merge_slot(d + k)] = op[k];
        }
    }
    __syncthreads();
    // lane-contiguous 16-byte stores: 4 consecutive outputs per thread and step (they never straddle a padding word)
#pragma unroll
    for (int q = 0; q < RK_TILE / (4 * RK_THREADS); ++q) {
        const int p = 4 * (q * RK_THREADS + static_cast<int>(threadIdx.x));
        const int s0 = merge_slot(p);
        if (p + 4 <= n) {
            *reinterpret_cast<uint4*>(key_out + o0 + p) = make_uint4(o_key[s0], o_key[s0 + 1], o_key[s0 + 2], o_key[s0 + 3]);
            *reinterpret_cast<uint4*>(pay_out + o0 + p) = make_uint4(o_pay[s0], o_pay[s0 + 1], o_pay[s0 + 2], o_pay[s0 + 3]);
        } else {
            for (int e = 0; p + e < n; ++e) {
                key_out[o0 + p + e] = o_key[s0 + e];
                pay_out[o0 + p + e] = o_pay[s0 + e];
            }
        }
    }
}

size_t rank_merge_ws_bytes(long long count) {
    const size_t split_bytes = static_cast<size_t>(rank_tiles(count) + 1) * sizeof(long long);
    return ((split_bytes + 255) & ~size_t(255)) + 256;              // Arena rounding + the alignment slack
}

int launch_rank_merge(const uint32_t* key_a, const uint32_t* pay_a, long long na, const uint32_t* key_b,
                      const uint32_t* pay_b, long long nb, uint32_t* key_out, uint32_t* pay_out, void* ws,
                      size_t ws_bytes, cudaStream_t st) {
    if (na + nb <= 0) return GCGCN_OK;
    Arena a = rank_arena(ws, ws_bytes);
    const int tiles = rank_tiles(na + nb);
    long long* split = a.take<long long>(tiles + 1);
    if (split == nullptr) return fail(GCGCN_ERR_WORKSPACE, "rank_merge: workspace too small (%zu bytes)", ws_bytes);
    merge_partition_kernel<<<ceil_div(tiles + 1, 256), 256, 0, st>>>(key_a, pay_a, na, key_b, pay_b, nb, tiles, split);
    GCGCN_CHECK_LAUNCH("rank_merge_partition");
    merge_tile_kernel<<<tiles, RK_THREADS, 0, st>>>(key_a, pay_a, na, key_b, pay_b, nb, split, key_out, pay_out);
    GCGCN_CHECK_LAUNCH("rank_merge_tile");
    return GCGCN_OK;
}

// ---- curve -------------------------------------------------------------------------------------------------------
// x = f32(c / T), y = f32(c / (k + 1)): one double division, rounded once.  f1 = 2 x y / ((x + y) + 1e-20) in float32,
// each operation rounded (no contraction): NumPy's  2 * pr_x * pr_y / (pr_x + pr_y + 1e-20)  on float32 arrays.
__device__ __forceinline__ float curve_ratio(long long a, long long b) {
    return __double2float_rn(static_cast<double>(a) / static_cast<double>(b));
}
__device__ __forceinline__ float curve_f1(float x, float y) {
    return __fdiv_rn(__fmul_rn(__fmul_rn(2.f, x), y), __fadd_rn(__fadd_rn(x, y), 1e-20f));
}
// Ign precision: facts seen in training are left out of the numerator and the denominator
__device__ __forceinline__ float curve_ign(long long c, long long t, long long k1) {
    return t == c ? 0.f : curve_ratio(c - t, k1 - t);
}
// one np.trapezoid term in float32:  (x1 - x0) * (y1 + y0) / 2
__device__ __forceinline__ double curve_trap(float x0, float x1, float y0, float y1) {
    return static_cast<double>(__fdiv_rn(__fmul_rn(__fsub_rn(x1, x0), __fadd_rn(y1, y0)), 2.f));
}

// per-tile packed flag counts: correct in the low word, correct & intrain in the high word (both < 2^30)
__global__ void __launch_bounds__(RK_THREADS)
curve_count_kernel(const uint32_t* __restrict__ pay, long long count, unsigned long long* __restrict__ flags) {
    __shared__ unsigned long long s_warp[33];
    const long long base = static_cast<long long>(blockIdx.x) * RK_TILE + threadIdx.x * static_cast<long long>(RK_IPT);
    uint32_t p[RK_IPT];
    load16(pay, base, count, p);
    unsigned long long acc = 0;
#pragma unroll
    for (int k = 0; k < RK_IPT; ++k) acc += (p[k] & 1u) + (static_cast<unsigned long long>((p[k] & 3u) == 3u) << 32);
    unsigned long long total;
    block_excl_scan<unsigned long long, RK_THREADS>(acc, s_warp, &total);
    if (threadIdx.x == 0) flags[blockIdx.x] = total;
}

// Tile `tile` of the run pay[0, count): thread t owns positions [tile TILE + 16 t, +16).  prefix = the scanned tile
// counts at `slot` + an in-tile scan; the tile's partials go to index `slot` of the output arrays.
// POINTS: write x, y (and yi with intrain) of every position instead of the tile's partials.
// SEGMENT: the run is one relation's segment of a partitioned ranking, with its first tile at slot `first`: its counts
// are the scanned counts minus those at `first`, and as it starts at any alignment the CTA stages its positions (and
// the next tile's first) in s_stage [RK_TILE + 4] with coalesced loads instead of 16-byte loads per thread.
template <bool POINTS, bool SEGMENT>
__device__ __forceinline__ void curve_main(const uint32_t* __restrict__ pay, long long count, long long T,
                                           int has_intrain, int tile, const unsigned long long* __restrict__ tile_prefix,
                                           long long first, uint32_t* __restrict__ s_stage, long long slot,
                                           float* __restrict__ best_f1, long long* __restrict__ best_pos,
                                           float* __restrict__ best_ign, double* __restrict__ auc,
                                           double* __restrict__ ign_auc, float* __restrict__ px,
                                           float* __restrict__ py, float* __restrict__ pyi) {
    __shared__ unsigned long long s_warp[33];
    __shared__ float s_f1[RK_THREADS], s_ign[RK_THREADS];
    __shared__ long long s_pos[RK_THREADS];
    __shared__ double s_auc[RK_THREADS], s_iauc[RK_THREADS];
    const long long base = static_cast<long long>(tile) * RK_TILE + threadIdx.x * static_cast<long long>(RK_IPT);
    uint32_t p[RK_IPT + 1];
    if constexpr (SEGMENT) {
        const long long t0 = static_cast<long long>(tile) * RK_TILE;
        for (int q = threadIdx.x; q < RK_TILE + 4; q += RK_THREADS) s_stage[q] = t0 + q < count ? pay[t0 + q] : 0u;
        __syncthreads();
        const uint4* s4 = reinterpret_cast<const uint4*>(s_stage + threadIdx.x * RK_IPT);
#pragma unroll
        for (int q = 0; q < RK_IPT / 4; ++q) reinterpret_cast<uint4*>(p)[q] = s4[q];
        p[RK_IPT] = s_stage[threadIdx.x * RK_IPT + RK_IPT];
    } else {
        load16(pay, base, count, *reinterpret_cast<uint32_t(*)[RK_IPT]>(p));
        p[RK_IPT] = base + RK_IPT < count ? pay[base + RK_IPT] : 0u;
    }
    unsigned long long acc = 0;
#pragma unroll
    for (int k = 0; k < RK_IPT; ++k) acc += (p[k] & 1u) + (static_cast<unsigned long long>((p[k] & 3u) == 3u) << 32);
    const unsigned long long pre = block_excl_scan<unsigned long long, RK_THREADS>(acc, s_warp, nullptr) +
                                   (SEGMENT ? tile_prefix[slot] - tile_prefix[first] : tile_prefix[slot]);
    long long c = static_cast<long long>(pre & 0xffffffffull), t = static_cast<long long>(pre >> 32);
    float f1_best = -1.f, ign_best = -1.f;
    long long pos_best = -1;
    double a = 0.0, ai = 0.0;
    // (x, y, yi) at position k carried to the trapezoid term of (k, k + 1)
    float xk = 0.f, yk = 0.f, yik = 0.f;
#pragma unroll
    for (int k = 0; k <= RK_IPT; ++k) {
        const long long pos = base + k;
        if (pos < count) {
            c += p[k] & 1u;
            t += (p[k] & 3u) == 3u;
            const float x = curve_ratio(c, T), y = curve_ratio(c, pos + 1);
            const float yi = has_intrain ? curve_ign(c, t, pos + 1) : 0.f;
            if (k > 0) {
                a += curve_trap(xk, x, yk, y);
                if (has_intrain) ai += curve_trap(xk, x, yik, yi);
            }
            if (POINTS && k < RK_IPT) {
                px[pos] = x;
                py[pos] = y;
                if (has_intrain) pyi[pos] = yi;
            }
            if (!POINTS && k < RK_IPT) { // k == RK_IPT is the next thread's first position: only the term is ours
                const float f = curve_f1(x, y);
                if (f > f1_best) { f1_best = f; pos_best = pos; }
                if (has_intrain) ign_best = fmaxf(ign_best, curve_f1(x, yi));
                xk = x; yk = y; yik = yi;
            }
        }
    }
    if (POINTS) return;
    s_f1[threadIdx.x] = f1_best;
    s_pos[threadIdx.x] = pos_best;
    s_ign[threadIdx.x] = ign_best;
    s_auc[threadIdx.x] = a;
    s_iauc[threadIdx.x] = ai;
    __syncthreads();
    for (int s = RK_THREADS / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) {
            const int o = threadIdx.x + s;
            // first argmax: on equal f1 the smaller position wins
            if (s_f1[o] > s_f1[threadIdx.x] || (s_f1[o] == s_f1[threadIdx.x] && s_pos[o] < s_pos[threadIdx.x])) {
                s_f1[threadIdx.x] = s_f1[o];
                s_pos[threadIdx.x] = s_pos[o];
            }
            s_ign[threadIdx.x] = fmaxf(s_ign[threadIdx.x], s_ign[o]);
            s_auc[threadIdx.x] += s_auc[o];
            s_iauc[threadIdx.x] += s_iauc[o];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        best_f1[slot] = s_f1[0];
        best_pos[slot] = s_pos[0];
        best_ign[slot] = s_ign[0];
        auc[slot] = s_auc[0];
        ign_auc[slot] = s_iauc[0];
    }
}

__global__ void __launch_bounds__(RK_THREADS)
curve_main_kernel(const uint32_t* __restrict__ pay, long long count, long long T, int has_intrain,
                  const unsigned long long* __restrict__ tile_prefix, float* __restrict__ best_f1,
                  long long* __restrict__ best_pos, float* __restrict__ best_ign, double* __restrict__ auc,
                  double* __restrict__ ign_auc) {
    curve_main<false, false>(pay, count, T, has_intrain, blockIdx.x, tile_prefix, 0, nullptr, blockIdx.x, best_f1,
                             best_pos, best_ign, auc, ign_auc, nullptr, nullptr, nullptr);
}

__global__ void __launch_bounds__(RK_THREADS)
curve_points_kernel(const uint32_t* __restrict__ pay, long long count, long long T, int has_intrain,
                    const unsigned long long* __restrict__ tile_prefix, float* __restrict__ x, float* __restrict__ y,
                    float* __restrict__ yi) {
    curve_main<true, false>(pay, count, T, has_intrain, blockIdx.x, tile_prefix, 0, nullptr, blockIdx.x, nullptr,
                            nullptr, nullptr, nullptr, nullptr, x, y, yi);
}

// One block: fixed-order reduction of the tile partials of the run key / pay [0, count), w, and the curve values at w.
// tile_prefix[t] - prefix_base = the flag counts before tile t of the run.
__device__ __forceinline__ void curve_finish(const uint32_t* __restrict__ key, const uint32_t* __restrict__ pay,
                                             long long count, long long T, int has_intrain, double input_theta,
                                             int tiles, const unsigned long long* __restrict__ tile_prefix,
                                             unsigned long long prefix_base, const float* __restrict__ best_f1,
                                             const long long* __restrict__ best_pos,
                                             const float* __restrict__ best_ign, const double* __restrict__ auc,
                                             const double* __restrict__ ign_auc, gcgcn_rank_result* __restrict__ res) {
    __shared__ float s_f1[1024], s_ign[1024];
    __shared__ long long s_pos[1024];
    __shared__ double s_auc[1024], s_iauc[1024];
    __shared__ long long s_w;
    __shared__ unsigned long long s_warp[33];
    float f = -1.f, g = -1.f;
    long long bp = -1;
    double a = 0.0, ai = 0.0;
    for (int i = threadIdx.x; i < tiles; i += 1024) {       // ascending tiles per thread: strict > keeps the first
        if (best_f1[i] > f) { f = best_f1[i]; bp = best_pos[i]; }
        g = fmaxf(g, best_ign[i]);
        a += auc[i];
        ai += ign_auc[i];
    }
    s_f1[threadIdx.x] = f; s_pos[threadIdx.x] = bp; s_ign[threadIdx.x] = g;
    s_auc[threadIdx.x] = a; s_iauc[threadIdx.x] = ai;
    __syncthreads();
    for (int s = 512; s > 0; s >>= 1) {
        if (threadIdx.x < s) {
            const int o = threadIdx.x + s;
            // equal f1: the smaller position wins (the tree does not keep positions in order)
            if (s_f1[o] > s_f1[threadIdx.x] || (s_f1[o] == s_f1[threadIdx.x] && s_pos[o] < s_pos[threadIdx.x])) {
                s_f1[threadIdx.x] = s_f1[o];
                s_pos[threadIdx.x] = s_pos[o];
            }
            s_ign[threadIdx.x] = fmaxf(s_ign[threadIdx.x], s_ign[o]);
            s_auc[threadIdx.x] += s_auc[o];
            s_iauc[threadIdx.x] += s_iauc[o];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        long long w;
        if (input_theta == -1.0) {
            w = s_pos[0];
        } else {
            // scores descend along the ranking: count the prefix with score > input_theta
            long long lo = 0, hi = count;
            while (lo < hi) {
                const long long mid = (lo + hi) >> 1;
                if (static_cast<double>(key_score(key[mid])) > input_theta) lo = mid + 1;
                else hi = mid;
            }
            w = lo > 0 ? lo - 1 : 0;
        }
        s_w = w;
    }
    __syncthreads();
    // flag counts up to and including w: the scanned tile prefix + this tile's positions <= w
    const long long w = s_w;
    const long long t0 = (w / RK_TILE) * RK_TILE;
    unsigned long long acc = 0;
    for (long long i = t0 + threadIdx.x; i <= w; i += 1024) {
        const uint32_t p = pay[i];
        acc += (p & 1u) + (static_cast<unsigned long long>((p & 3u) == 3u) << 32);
    }
    unsigned long long total;
    block_excl_scan<unsigned long long, 1024>(acc, s_warp, &total);
    if (threadIdx.x == 0) {
        const unsigned long long pre = total + (tile_prefix[w / RK_TILE] - prefix_base);
        const long long c = static_cast<long long>(pre & 0xffffffffull), t = static_cast<long long>(pre >> 32);
        const float x = curve_ratio(c, T), y = curve_ratio(c, w + 1);
        gcgcn_rank_result r;
        r.count = count;
        r.total_recall = T;
        r.best_pos = s_pos[0];
        r.w = w;
        r.auc = s_auc[0];
        r.ign_auc = has_intrain ? s_iauc[0] : 0.0;
        r.f1 = s_f1[0];
        r.theta = key_score(key[s_pos[0]]);
        r.f1_at_w = curve_f1(x, y);
        r.precision_at_w = y;
        r.recall_at_w = x;
        r.ign_f1 = has_intrain ? s_ign[0] : 0.f;
        r.ign_f1_at_w = has_intrain ? curve_f1(x, curve_ign(c, t, w + 1)) : 0.f;
        r.reserved = 0;
        *res = r;
    }
}

__global__ void __launch_bounds__(1024)
curve_finish_kernel(const uint32_t* __restrict__ key, const uint32_t* __restrict__ pay, long long count, long long T,
                    int has_intrain, double input_theta, int tiles, const unsigned long long* __restrict__ tile_prefix,
                    const float* __restrict__ best_f1, const long long* __restrict__ best_pos,
                    const float* __restrict__ best_ign, const double* __restrict__ auc,
                    const double* __restrict__ ign_auc, gcgcn_rank_result* __restrict__ res) {
    curve_finish(key, pay, count, T, has_intrain, input_theta, tiles, tile_prefix, 0ull, best_f1, best_pos, best_ign,
                 auc, ign_auc, res);
}

int launch_rank_curve(const uint32_t* key, const uint32_t* pay, long long count, long long T, int has_intrain,
                      double input_theta, gcgcn_rank_result* res, void* ws, size_t ws_bytes, cudaStream_t st) {
    Arena a = rank_arena(ws, ws_bytes);
    CurveWs w;
    if (!curve_ws_take(a, count, &w)) return fail(GCGCN_ERR_WORKSPACE, "rank_curve: workspace too small (%zu bytes)", ws_bytes);
    const int tiles = rank_tiles(count);
    curve_count_kernel<<<tiles, RK_THREADS, 0, st>>>(pay, count, w.flags);
    GCGCN_CHECK_LAUNCH("rank_curve_count");
    GCGCN_TRY(launch_scan<unsigned long long>(w.flags, tiles, w.sums, st));
    curve_main_kernel<<<tiles, RK_THREADS, 0, st>>>(pay, count, T, has_intrain, w.flags, w.best_f1, w.best_pos,
                                                    w.best_ign, w.auc, w.ign_auc);
    GCGCN_CHECK_LAUNCH("rank_curve_main");
    curve_finish_kernel<<<1, 1024, 0, st>>>(key, pay, count, T, has_intrain, input_theta, tiles, w.flags, w.best_f1,
                                            w.best_pos, w.best_ign, w.auc, w.ign_auc, res);
    GCGCN_CHECK_LAUNCH("rank_curve_finish");
    return GCGCN_OK;
}

int launch_rank_curve_points(const uint32_t* pay, long long count, long long T, int has_intrain, float* x, float* y,
                             float* yi, void* ws, size_t ws_bytes, cudaStream_t st) {
    Arena a = rank_arena(ws, ws_bytes);
    CurveWs w;
    if (!curve_ws_take(a, count, &w))
        return fail(GCGCN_ERR_WORKSPACE, "rank_curve_points: workspace too small (%zu bytes)", ws_bytes);
    const int tiles = rank_tiles(count);
    curve_count_kernel<<<tiles, RK_THREADS, 0, st>>>(pay, count, w.flags);
    GCGCN_CHECK_LAUNCH("rank_curve_count");
    GCGCN_TRY(launch_scan<unsigned long long>(w.flags, tiles, w.sums, st));
    curve_points_kernel<<<tiles, RK_THREADS, 0, st>>>(pay, count, T, has_intrain, w.flags, x, y, yi);
    GCGCN_CHECK_LAUNCH("rank_curve_points");
    return GCGCN_OK;
}

// ---- per relation ------------------------------------------------------------------------------------------------
// Every document gives n^2 - n candidates to each relation and its first id is a multiple of R - 1, so a candidate's
// relation is (id mod (R - 1)) + 1 and every relation holds L = count / (R - 1) candidates.  The stable partition of a
// ranking by relation (one more radix pass, digit from the payload) puts relation r's candidates, in ranked order, at
// [(r - 1) L, r L).  The per-relation curve tiles every segment from its own start (blockIdx.y = r - 1, blockIdx.x =
// tile of the segment), so no tile spans two relations: (R - 1) ceil(L / TILE) <= tiles + R - 1 pieces, and the flag
// counts of a segment are the scanned piece counts minus the value at its first piece.
int launch_rank_by_relation(const uint32_t* key, const uint32_t* pay, long long count, int R, uint32_t* rel_key,
                            uint32_t* rel_pay, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (R == 2) {                                            // one relation: the partition is the ranking
        GCGCN_TRY(cuda_ok(cudaMemcpyAsync(rel_key, key, count * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st),
                          "rank_by_relation"));
        return cuda_ok(cudaMemcpyAsync(rel_pay, pay, count * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st),
                       "rank_by_relation");
    }
    Arena a = rank_arena(ws, ws_bytes);
    const int tiles = rank_tiles(count);
    const long long ncounts = static_cast<long long>(tiles) * RK_RADIX;
    uint32_t* counts = a.take<uint32_t>(ncounts);
    uint32_t* sums = a.take<uint32_t>(ceil_div(ncounts, SCAN_CHUNK));
    if (counts == nullptr || sums == nullptr)
        return fail(GCGCN_ERR_WORKSPACE, "rank_by_relation: workspace too small (%zu bytes)", ws_bytes);
    radix_upsweep_kernel<DIGIT_RELATION><<<tiles, RK_THREADS, 0, st>>>(pay, count, R - 1, tiles, counts);
    GCGCN_CHECK_LAUNCH("rank_relation_upsweep");
    GCGCN_TRY(launch_scan<uint32_t>(counts, ncounts, sums, st));
    radix_downsweep_kernel<DIGIT_RELATION><<<tiles, RK_THREADS, 0, st>>>(key, pay, count, R - 1, tiles, counts, rel_key,
                                                                        rel_pay);
    GCGCN_CHECK_LAUNCH("rank_relation_downsweep");
    return GCGCN_OK;
}

// T of segment s: the caller's value, or the segment's correct candidates (flags holds the exclusive scan of the
// piece counts, one entry past the last piece); < 1 means 1
__device__ __forceinline__ long long segment_recall(const long long* __restrict__ total_recall,
                                                    const unsigned long long* __restrict__ flags, int s,
                                                    int seg_tiles) {
    const long long v = total_recall != nullptr
                            ? total_recall[s]
                            : static_cast<long long>((flags[static_cast<long long>(s + 1) * seg_tiles] -
                                                      flags[static_cast<long long>(s) * seg_tiles]) & 0xffffffffull);
    return v < 1 ? 1 : v;
}

// packed flag counts of every piece (as curve_count_kernel, from coalesced loads of the segment); block (0, 0) also
// zeroes the entry past the last piece, so that the scan leaves the grand total there
__global__ void __launch_bounds__(RK_THREADS)
rel_curve_count_kernel(const uint32_t* __restrict__ pay, long long L, int seg_tiles,
                       unsigned long long* __restrict__ flags) {
    __shared__ unsigned long long s_warp[33];
    const uint32_t* run = pay + static_cast<long long>(blockIdx.y) * L;
    const long long t0 = static_cast<long long>(blockIdx.x) * RK_TILE;
    const int n = static_cast<int>(min(static_cast<long long>(RK_TILE), L - t0));
    unsigned long long acc = 0;
    for (int q = threadIdx.x; q < n; q += RK_THREADS) {
        const uint32_t p = run[t0 + q];
        acc += (p & 1u) + (static_cast<unsigned long long>((p & 3u) == 3u) << 32);
    }
    unsigned long long total;
    block_excl_scan<unsigned long long, RK_THREADS>(acc, s_warp, &total);
    if (threadIdx.x == 0) {
        flags[static_cast<long long>(blockIdx.y) * seg_tiles + blockIdx.x] = total;
        if (blockIdx.x == 0 && blockIdx.y == 0) flags[static_cast<long long>(gridDim.y) * seg_tiles] = 0ull;
    }
}

__global__ void __launch_bounds__(RK_THREADS)
rel_curve_main_kernel(const uint32_t* __restrict__ pay, long long L, int seg_tiles,
                      const long long* __restrict__ total_recall, int has_intrain,
                      const unsigned long long* __restrict__ flags, float* __restrict__ best_f1,
                      long long* __restrict__ best_pos, float* __restrict__ best_ign, double* __restrict__ auc,
                      double* __restrict__ ign_auc) {
    __shared__ __align__(16) uint32_t s_stage[RK_TILE + 4];
    const int s = blockIdx.y;
    const long long first = static_cast<long long>(s) * seg_tiles, slot = first + blockIdx.x;
    curve_main<false, true>(pay + s * L, L, segment_recall(total_recall, flags, s, seg_tiles), has_intrain, blockIdx.x,
                            flags, first, s_stage, slot, best_f1, best_pos, best_ign, auc, ign_auc, nullptr, nullptr,
                            nullptr);
}

// one block per relation: curve_finish over the segment's pieces, in tile order
__global__ void __launch_bounds__(1024)
rel_curve_finish_kernel(const uint32_t* __restrict__ key, const uint32_t* __restrict__ pay, long long L, int seg_tiles,
                        const long long* __restrict__ total_recall, int has_intrain,
                        const double* __restrict__ input_theta, const unsigned long long* __restrict__ flags,
                        const float* __restrict__ best_f1, const long long* __restrict__ best_pos,
                        const float* __restrict__ best_ign, const double* __restrict__ auc,
                        const double* __restrict__ ign_auc, gcgcn_rank_result* __restrict__ res) {
    const int s = blockIdx.x;
    const long long first = static_cast<long long>(s) * seg_tiles;
    curve_finish(key + s * L, pay + s * L, L, segment_recall(total_recall, flags, s, seg_tiles), has_intrain,
                 input_theta[s], seg_tiles, flags + first, flags[first], best_f1 + first, best_pos + first,
                 best_ign + first, auc + first, ign_auc + first, res + s);
}

struct RelCurveWs {
    unsigned long long *flags, *sums;
    float *best_f1, *best_ign;
    long long* best_pos;
    double *auc, *ign_auc;
};
static int seg_tiles_of(long long count, int R) { return rank_tiles(count / (R - 1)); }
static bool rel_curve_ws_take(Arena& a, long long count, int R, RelCurveWs* w) {
    const long long pieces = static_cast<long long>(R - 1) * seg_tiles_of(count, R);
    w->flags = a.take<unsigned long long>(pieces + 1);
    w->sums = a.take<unsigned long long>(ceil_div(pieces + 1, SCAN_CHUNK));
    w->best_f1 = a.take<float>(pieces);
    w->best_ign = a.take<float>(pieces);
    w->best_pos = a.take<long long>(pieces);
    w->auc = a.take<double>(pieces);
    w->ign_auc = a.take<double>(pieces);
    return w->flags && w->sums && w->best_f1 && w->best_ign && w->best_pos && w->auc && w->ign_auc;
}

int launch_rank_curve_relations(const uint32_t* key, const uint32_t* pay, long long count, int R,
                                const long long* total_recall, int has_intrain, const double* input_theta,
                                gcgcn_rank_result* res, void* ws, size_t ws_bytes, cudaStream_t st) {
    Arena a = rank_arena(ws, ws_bytes);
    RelCurveWs w;
    if (!rel_curve_ws_take(a, count, R, &w))
        return fail(GCGCN_ERR_WORKSPACE, "rank_curve_relations: workspace too small (%zu bytes)", ws_bytes);
    const long long L = count / (R - 1);
    const int seg_tiles = seg_tiles_of(count, R);
    const dim3 grid(seg_tiles, R - 1);
    rel_curve_count_kernel<<<grid, RK_THREADS, 0, st>>>(pay, L, seg_tiles, w.flags);
    GCGCN_CHECK_LAUNCH("rank_relation_curve_count");
    GCGCN_TRY(launch_scan<unsigned long long>(w.flags, static_cast<long long>(R - 1) * seg_tiles + 1, w.sums, st));
    rel_curve_main_kernel<<<grid, RK_THREADS, 0, st>>>(pay, L, seg_tiles, total_recall, has_intrain, w.flags,
                                                       w.best_f1, w.best_pos, w.best_ign, w.auc, w.ign_auc);
    GCGCN_CHECK_LAUNCH("rank_relation_curve_main");
    rel_curve_finish_kernel<<<R - 1, 1024, 0, st>>>(key, pay, L, seg_tiles, total_recall, has_intrain, input_theta,
                                                    w.flags, w.best_f1, w.best_pos, w.best_ign, w.auc, w.ign_auc, res);
    GCGCN_CHECK_LAUNCH("rank_relation_curve_finish");
    return GCGCN_OK;
}

// ---- selection at one threshold per relation -----------------------------------------------------------------------
// A ranked candidate is selected when its score > theta[relation - 1].  Per tile: counts of (selected) and of (selected
// and correct | selected, correct and intrain << 32) -> two exclusive scans (one entry past the last tile holds the
// totals) -> a stable in-tile compaction of the selected (key, payload) pairs.
__device__ __forceinline__ void load_theta(const float* __restrict__ theta, int rm1, float* s_theta) {
    for (int r = threadIdx.x; r < rm1; r += RK_THREADS) s_theta[r] = theta[r];
    __syncthreads();
}

__global__ void __launch_bounds__(RK_THREADS)
select_count_kernel(const uint32_t* __restrict__ key, const uint32_t* __restrict__ pay, long long count, int rm1,
                    const float* __restrict__ theta, int tiles, uint32_t* __restrict__ sel,
                    unsigned long long* __restrict__ flags) {
    __shared__ float s_theta[RK_RADIX];
    __shared__ uint32_t s_warp[33];
    __shared__ unsigned long long s_warp64[33];
    load_theta(theta, rm1, s_theta);
    const long long base = static_cast<long long>(blockIdx.x) * RK_TILE + threadIdx.x * static_cast<long long>(RK_IPT);
    uint32_t k[RK_IPT], p[RK_IPT];
    load16(key, base, count, k);
    load16(pay, base, count, p);
    uint32_t m = 0;
    unsigned long long ct = 0;
#pragma unroll
    for (int q = 0; q < RK_IPT; ++q) {
        if (base + q < count && key_score(k[q]) > s_theta[(p[q] >> 2) % static_cast<uint32_t>(rm1)]) {
            ++m;
            ct += (p[q] & 1u) + (static_cast<unsigned long long>((p[q] & 3u) == 3u) << 32);
        }
    }
    uint32_t m_total;
    unsigned long long ct_total;
    block_excl_scan<uint32_t, RK_THREADS>(m, s_warp, &m_total);
    block_excl_scan<unsigned long long, RK_THREADS>(ct, s_warp64, &ct_total);
    if (threadIdx.x == 0) {
        sel[blockIdx.x] = m_total;
        flags[blockIdx.x] = ct_total;
        if (blockIdx.x == 0) { sel[tiles] = 0u; flags[tiles] = 0ull; }
    }
}

__global__ void __launch_bounds__(RK_THREADS)
select_scatter_kernel(const uint32_t* __restrict__ key, const uint32_t* __restrict__ pay, long long count, int rm1,
                      const float* __restrict__ theta, int tiles, const uint32_t* __restrict__ sel,
                      const unsigned long long* __restrict__ flags, uint32_t* __restrict__ out_key,
                      uint32_t* __restrict__ out_pay, long long* __restrict__ counts) {
    __shared__ float s_theta[RK_RADIX];
    __shared__ uint32_t s_warp[33];
    load_theta(theta, rm1, s_theta);
    const long long base = static_cast<long long>(blockIdx.x) * RK_TILE + threadIdx.x * static_cast<long long>(RK_IPT);
    uint32_t k[RK_IPT], p[RK_IPT];
    load16(key, base, count, k);
    load16(pay, base, count, p);
    uint32_t pick = 0, m = 0;
#pragma unroll
    for (int q = 0; q < RK_IPT; ++q) {
        const bool on = base + q < count && key_score(k[q]) > s_theta[(p[q] >> 2) % static_cast<uint32_t>(rm1)];
        pick |= (on ? 1u : 0u) << q;
        m += on;
    }
    long long o = block_excl_scan<uint32_t, RK_THREADS>(m, s_warp, nullptr) + static_cast<long long>(sel[blockIdx.x]);
#pragma unroll
    for (int q = 0; q < RK_IPT; ++q) {
        if ((pick >> q) & 1u) {
            out_key[o] = k[q];
            out_pay[o] = p[q];
            ++o;
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        counts[0] = sel[tiles];
        counts[1] = static_cast<long long>(flags[tiles] & 0xffffffffull);
        counts[2] = static_cast<long long>(flags[tiles] >> 32);
    }
}

struct SelectWs {
    uint32_t *sel, *sel_sums;
    unsigned long long *flags, *sums;
};
static bool select_ws_take(Arena& a, long long count, SelectWs* w) {
    const long long n = rank_tiles(count) + 1;
    w->sel = a.take<uint32_t>(n);
    w->sel_sums = a.take<uint32_t>(ceil_div(n, SCAN_CHUNK));
    w->flags = a.take<unsigned long long>(n);
    w->sums = a.take<unsigned long long>(ceil_div(n, SCAN_CHUNK));
    return w->sel && w->sel_sums && w->flags && w->sums;
}

int launch_rank_select(const uint32_t* key, const uint32_t* pay, long long count, int R, const float* theta,
                       uint32_t* out_key, uint32_t* out_pay, long long* counts, void* ws, size_t ws_bytes,
                       cudaStream_t st) {
    Arena a = rank_arena(ws, ws_bytes);
    SelectWs w;
    if (!select_ws_take(a, count, &w))
        return fail(GCGCN_ERR_WORKSPACE, "rank_select: workspace too small (%zu bytes)", ws_bytes);
    const int tiles = rank_tiles(count);
    select_count_kernel<<<tiles, RK_THREADS, 0, st>>>(key, pay, count, R - 1, theta, tiles, w.sel, w.flags);
    GCGCN_CHECK_LAUNCH("rank_select_count");
    GCGCN_TRY(launch_scan<uint32_t>(w.sel, tiles + 1, w.sel_sums, st));
    GCGCN_TRY(launch_scan<unsigned long long>(w.flags, tiles + 1, w.sums, st));
    select_scatter_kernel<<<tiles, RK_THREADS, 0, st>>>(key, pay, count, R - 1, theta, tiles, w.sel, w.flags, out_key,
                                                        out_pay, counts);
    GCGCN_CHECK_LAUNCH("rank_select_scatter");
    return GCGCN_OK;
}

size_t rank_relations_ws_bytes(long long count, int R) {
    if (count <= 0 || R < 2) return 512;
    const long long tiles = rank_tiles(count), ncounts = tiles * RK_RADIX;
    const size_t partition = ((ncounts * sizeof(uint32_t) + 255) & ~size_t(255)) +
                             ((ceil_div(ncounts, SCAN_CHUNK) * sizeof(uint32_t) + 255) & ~size_t(255));
    Arena probe(reinterpret_cast<void*>(256), ~size_t(0) >> 1);
    RelCurveWs c;
    rel_curve_ws_take(probe, count, R, &c);
    Arena probe2(reinterpret_cast<void*>(256), ~size_t(0) >> 1);
    SelectWs s;
    select_ws_take(probe2, count, &s);
    return std::max(partition, std::max(probe.off, probe2.off)) + 256;
}

// ---- decode -----------------------------------------------------------------------------------------------------
// doc_off [docs + 1]: first candidate id of every document (in add() order); the document of an id is the last one
// whose offset is <= id (documents with n <= 1 own no ids and share their successor's offset).
__global__ void __launch_bounds__(256)
rank_decode_kernel(const uint32_t* __restrict__ key, const uint32_t* __restrict__ pay, long long rows,
                   const long long* __restrict__ doc_off, const int* __restrict__ doc_n, int docs, int R,
                   int* __restrict__ doc, int* __restrict__ row, int* __restrict__ col, int* __restrict__ rel,
                   float* __restrict__ score) {
    const long long k = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (k >= rows) return;
    const long long id = pay[k] >> 2;
    int lo = 0, hi = docs;                           // first document whose offset is > id, minus one
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (doc_off[mid] <= id) lo = mid + 1;
        else hi = mid;
    }
    const int b = lo - 1;
    const int n = doc_n[b];
    const long long local = id - doc_off[b];
    const long long per_row = static_cast<long long>(n - 1) * (R - 1);
    const int i = static_cast<int>(local / per_row);
    const long long rem = local - i * per_row;
    const int jj = static_cast<int>(rem / (R - 1));
    doc[k] = b;
    row[k] = i;
    col[k] = jj + (jj >= i);
    rel[k] = static_cast<int>(rem - static_cast<long long>(jj) * (R - 1)) + 1;
    score[k] = key_score(key[k]);
}

int launch_rank_decode(const uint32_t* key, const uint32_t* pay, long long rows, const long long* doc_off,
                       const int* doc_n, int docs, int R, int* doc, int* row, int* col, int* rel, float* score,
                       cudaStream_t st) {
    if (rows <= 0) return GCGCN_OK;
    rank_decode_kernel<<<ceil_div(rows, 256), 256, 0, st>>>(key, pay, rows, doc_off, doc_n, docs, R, doc, row, col, rel,
                                                           score);
    GCGCN_CHECK_LAUNCH("rank_decode");
    return GCGCN_OK;
}

}  // namespace gcgcn
