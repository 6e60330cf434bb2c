// tcgen05 / TMEM projection GEMM with fp32-accurate "3xTF32" operand splitting (sm_100a).
//
//   C[M,N] = alpha * op(A)[M,K] * op(B)[K,N] + beta * C + bias          (row-major fp32 in HBM)
//
// Why this shape of kernel: the dense contractions of the path are (all node rows of the batch) x
// (128..1024)-wide projections and their transposes.  fp32 parity with the reference (<= 1e-4 abs)
// rules out single-pass TF32 (10-bit mantissa), so every fp32 operand value a is split on the fly into
//   a_hi = a with the low 13 mantissa bits cleared (exactly representable in TF32)
//   a_lo = a - a_hi                                  (exact in fp32; the MMA keeps its top 11 bits)
// and the product is accumulated as  A_lo*B_hi + A_hi*B_lo + A_hi*B_hi  (error ~2^-20 relative) by
// three tcgen05.mma.kind::tf32 instructions per K-step into one fp32 accumulator in TMEM.
//
// Structure (one CTA per SM, persistent over 128x128 output tiles):
//   warps 0-15 producers (4 groups of 4 warps, one K block each in flight): global -> registers -> {hi,lo} split -> shared memory in the UMMA
//              canonical K-major no-swizzle layout ([K/4][128 rows][16 B]); operands stored
//              "transposed" in HBM (MN-contiguous) are transposed in registers on the way, so the
//              tensor core always sees K-major tiles.  TMA cannot be used for this stage because the
//              split is arithmetic on every element.
//   warp 16    allocates TMEM, then one elected lane issues the MMAs and commits them to mbarriers
//   warps 17-20 epilogue: tcgen05.ld the 128x128 fp32 accumulator, apply alpha/beta/bias, store
// Pipelines: 3 shared-memory stages (full/empty mbarriers), 2 TMEM accumulators (tile i+1 is
// multiplied while tile i is stored).  K may be split across CTAs (weight gradients reduce over all
// node rows); partials go to the workspace and are reduced by splitk_reduce (deterministic).
#include "common.cuh"
#include "tc_ptx.cuh"

namespace gcgcn {

constexpr int TC_BM = 128, TC_BN = 128, TC_BK = 32, TC_STAGES = 3;
// One operand part = 8 K-chunk planes of [128 rows][16 B]; each plane is padded by 16 B so that a quarter
// warp storing the 8 chunks of one row (lanes = chunks) hits 8 different 16-byte bank groups.
constexpr int TC_PLANE_BYTES = 128 * 16 + 16;               // UMMA leading (K) byte offset (odd multiple of 16 B)
constexpr int TC_PART_BYTES = (TC_BK / 4) * TC_PLANE_BYTES; // one 128 x 32 fp32 operand part
constexpr int TC_STAGE_BYTES = 4 * TC_PART_BYTES;           // A_hi, A_lo, B_hi, B_lo
// epilogue transpose buffer: [32 rows][32 floats] per warp, the 16-byte chunk index XOR-swizzled with (row & 7) so that
// both the row-per-lane stores and the 8-lanes-per-row loads are bank-conflict free without padding
constexpr int TC_EPI_WARP_FLOATS = 32 * 32;
constexpr int TC_EPI_BYTES = 4 * TC_EPI_WARP_FLOATS * 4;
// GROUPS producer groups of 4 warps (one K block of global loads in flight each), then 1 MMA warp, then 4
// epilogue warps (warp index 4*GROUPS+1.. so that warp % 4 covers the TMEM lane quarters 1,2,3,0).
// Three groups, except on the presplit-A route: two there, because its producers double-buffer the scalar-loaded
// generated operand and need more registers per thread (128) than a 17-warp CTA leaves.
constexpr int tc_threads(int groups) { return (4 * groups + 5) * 32; }
constexpr int TC_TMEM_COLS = 256;                           // 2 accumulators x 128 fp32 columns
constexpr size_t TC_SMEM_BYTES = size_t(TC_STAGES) * TC_STAGE_BYTES + TC_EPI_BYTES + 1024 /*align*/ + 256 /*barriers*/;

struct TcArgs {
    int M, N, K, lda, ldb, ldc;
    const float* A;
    const float* B;
    const float* bias;
    float* C;
    float* partial;     // != nullptr -> split-K partial output [k_splits][M][N]
    float alpha, beta;
    int tiles_m, tiles_n, k_splits, k_per_split;
    const uint8_t* Bpre;            // != nullptr -> B operand pre-split into ready-to-copy stage blobs [tiles_n][kblocks]
    const uint8_t* Apre;            // != nullptr -> A operand pre-split likewise, blobs [tiles_m][kblocks]
    int kblocks;                    // ceil(K / TC_BK), blob index stride of Bpre
    int batch;                      // independent products per launch (same shapes, strided operands)
    long long sA, sB, sC;           // element strides between consecutive products
    // row-dot epilogue (gemm_tc_tmema_kernel<1>): instead of storing the 128 x 128 tile, every row is contracted with
    // the matching 128 values of rd_t: rd_out[(tile_n * 2 + half) * rd_ld + row] = sum_{c in half} acc[row][c] rd_t[row][c]
    const float* rd_t;              // [M][128]
    float* rd_out;                  // [tiles_n][2][rd_ld]
    long long rd_ld;
    // row-accumulate epilogue (gemm_tc_tmema_kernel<2>): rd_out[row][c] = sum_nt rd_t[row * rd_ld + nt] * acc_nt[row][c]
    // (rd_t is then a [M][rd_ld] matrix of per-(row, column tile) weights, rd_out a [M][128] matrix)
    // generated B operand of the APRE path: column tile nt of op(B) is  bscale[k * lds + nt] * B[k][0..127]
    // (B a [K, 128] matrix shared by all column tiles) -- the Khatri-Rao factor of the bilinear weight gradient
    const float* bscale;
    int lds;
    // seq_k != 0 (APRE path, partial == nullptr): the k_splits K ranges of a tile are walked by ONE CTA in order
    // (grid = tiles), each accumulated in TMEM from zero and added into C by the epilogue (beta = 1 after the first).
    // Bounds the length of a single tensor-core accumulation: its fp32 adds truncate, and over tens of thousands of
    // K steps the bias reaches 1e-4 of the result.
    int seq_k;
};

// PTX wrappers: tc_ptx.cuh

// UMMA shared-memory descriptor, K-major, no swizzle: 8-row x 16-byte core matrices are 128 contiguous
// bytes; the next core matrix along M/N is 128 B away (SBO), the next along K is one padded chunk plane
// (TC_PLANE_BYTES) away (LBO).
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
    uint64_t d = (smem_addr >> 4) & 0x3FFFu;
    d |= static_cast<uint64_t>(TC_PLANE_BYTES >> 4) << 16;   // leading (K) byte offset
    d |= static_cast<uint64_t>(128 >> 4) << 32;          // stride (M/N) byte offset
    d |= static_cast<uint64_t>(1) << 46;                 // descriptor version (Blackwell)
    return d;
}
// kind::tf32, fp32 accumulate, A and B K-major, N = 128, M = 128
constexpr uint32_t TC_IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((TC_BN >> 3) << 17) | ((TC_BM >> 4) << 24);

__device__ __forceinline__ void split_store(float* hi_base, float* lo_base, int chunk, int row, float4 a) {
    float4 h, l;
    h.x = __uint_as_float(__float_as_uint(a.x) & 0xffffe000u);
    h.y = __uint_as_float(__float_as_uint(a.y) & 0xffffe000u);
    h.z = __uint_as_float(__float_as_uint(a.z) & 0xffffe000u);
    h.w = __uint_as_float(__float_as_uint(a.w) & 0xffffe000u);
    l.x = a.x - h.x; l.y = a.y - h.y; l.z = a.z - h.z; l.w = a.w - h.w;
    const int off = chunk * (TC_PLANE_BYTES / 4) + row * 4;
    *reinterpret_cast<float4*>(hi_base + off) = h;
    *reinterpret_cast<float4*>(lo_base + off) = l;
}

// One 128(rows) x 32(k) operand tile = 1024 float4; each of the 128 threads of a producer group moves 8.
// Thread -> (row, 16-byte K chunk) assignment of its i-th float4:
//   K-contiguous source: a warp instruction covers 4 consecutive rows x all 8 chunks, so global loads
//     are 4 fully used 128-byte lines and the shared-memory stores (rows 16 B apart, chunk planes
//     2 KB + 16 B apart) spread over all 32 banks (4 wavefronts for 512 B, the minimum);
//   MN-contiguous source (transposed in registers): lanes walk rows, so the 4-byte global loads coalesce
//     into 128-byte lines and each store instruction writes 512 contiguous bytes.
template <bool KCONTIG>
__device__ __forceinline__ void tile_coord(int tid, int i, int& row, int& chunk) {
    if (KCONTIG) {
        const int w = tid >> 5, l = tid & 31;
        row = 32 * w + 4 * i + (l >> 3);
        chunk = l & 7;
    } else {
        row = tid;
        chunk = i;
    }
}

// KCONTIG: element (row, k) at src[row*ld + k]; otherwise at src[k*ld + row].  Out of range -> 0.
template <bool KCONTIG>
__device__ __forceinline__ void fetch_operand(const float* __restrict__ src, int ld, int row0, int rows_total,
                                              int k0, int kend, bool vec_ok, int tid, float4 (&v)[8]) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        int r, c;
        tile_coord<KCONTIG>(tid, i, r, c);
        const int row = row0 + r, k = k0 + 4 * c;
        const bool row_ok = row < rows_total;
        if (KCONTIG) {
            const float* p = src + static_cast<size_t>(row) * ld + k;
            if (row_ok && vec_ok && k + 4 <= kend) {
                v[i] = *reinterpret_cast<const float4*>(p);
            } else {
                float t[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) t[q] = (row_ok && k + q < kend) ? p[q] : 0.f;
                v[i] = make_float4(t[0], t[1], t[2], t[3]);
            }
        } else {
            float t[4];
#pragma unroll
            for (int q = 0; q < 4; ++q)
                t[q] = (row_ok && k + q < kend) ? src[static_cast<size_t>(k + q) * ld + row] : 0.f;
            v[i] = make_float4(t[0], t[1], t[2], t[3]);
        }
    }
}

template <bool KCONTIG>
__device__ __forceinline__ void store_operand(float* hi, float* lo, int tid, const float4 (&v)[8]) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        int r, c;
        tile_coord<KCONTIG>(tid, i, r, c);
        split_store(hi, lo, c, r, v[i]);
    }
}

// ---- MN-major operand tiles (both operands of a weight gradient C = A^T B are stored [K][MN], MN contiguous) -------
// The tensor core reads 32-bit operands in MN-major form through exactly one shared-memory layout, "128-byte swizzle
// with 32-byte base": column blocks of [k rows][32 mn] fp32, rows 128 B apart, the 32-byte chunk index XORed with
// (k % 4).  That is the operand's own row-major layout up to the XOR, so a K block is moved by coalesced 16-byte
// loads and 16-byte stores with no transposition in registers (the K-major route above pays 4-byte loads for it).
// One [32 k][128 mn] part = 4 column blocks of 4096 B; the four parts of a stage sit at multiples of 16 KB.
constexpr int TC_MN_BLOCK_BYTES = TC_BK * 128;              // one [32 k][32 mn] column block
constexpr int TC_MN_PART_BYTES = 4 * TC_MN_BLOCK_BYTES;     // 16 KB
static_assert(4 * TC_MN_PART_BYTES <= TC_STAGE_BYTES, "MN-major parts fit a stage");
__device__ __forceinline__ uint64_t make_desc_mn(uint32_t smem_addr) {
    uint64_t d = (smem_addr >> 4) & 0x3FFFu;
    d |= static_cast<uint64_t>(TC_MN_BLOCK_BYTES >> 4) << 16;   // leading byte offset: the next 32-wide column block
    d |= static_cast<uint64_t>(512 >> 4) << 32;                 // stride byte offset: the next atom of 4 k rows
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(1) << 61;                        // SWIZZLE_128B_BASE32B
    return d;
}
constexpr uint32_t TC_IDESC_MN = TC_IDESC | (1u << 15) | (1u << 16);   // A and B MN-major
// thread -> (k row, 16-byte chunk) of its i-th float4: warp w of the group owns column block w, a warp instruction
// covers 4 k rows x 128 B (four whole lines in HBM, 512 contiguous bytes in shared memory)
__device__ __forceinline__ void fetch_operand_mn(const float* __restrict__ src, int ld, int mn0, int mn_total, int k0, int kend,
                                                 bool vec_ok, int tid, float4 (&v)[8]) {
    const int w = tid >> 5, l = tid & 31;
    const int mn = mn0 + 32 * w + 4 * (l & 7);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int k = k0 + 4 * i + (l >> 3);
        const float* p = src + static_cast<size_t>(k) * ld + mn;
        if (k < kend && vec_ok && mn + 4 <= mn_total) {
            v[i] = *reinterpret_cast<const float4*>(p);
        } else {
            float t[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) t[q] = (k < kend && mn + q < mn_total) ? p[q] : 0.f;
            v[i] = make_float4(t[0], t[1], t[2], t[3]);
        }
    }
}
__device__ __forceinline__ void store_operand_mn(uint8_t* hi, uint8_t* lo, int tid, const float4 (&v)[8]) {
    const int w = tid >> 5, l = tid & 31, c = l & 7;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int krow = 4 * i + (l >> 3);
        const int off = w * TC_MN_BLOCK_BYTES + krow * 128 + (((((c >> 1) ^ (krow & 3)) << 1) | (c & 1)) << 4);
        const float4 a = v[i];
        float4 h, lw;
        h.x = __uint_as_float(__float_as_uint(a.x) & 0xffffe000u);
        h.y = __uint_as_float(__float_as_uint(a.y) & 0xffffe000u);
        h.z = __uint_as_float(__float_as_uint(a.z) & 0xffffe000u);
        h.w = __uint_as_float(__float_as_uint(a.w) & 0xffffe000u);
        lw.x = a.x - h.x; lw.y = a.y - h.y; lw.z = a.z - h.z; lw.w = a.w - h.w;
        *reinterpret_cast<float4*>(hi + off) = h;
        *reinterpret_cast<float4*>(lo + off) = lw;
    }
}

// Epilogue of one 128 x 128 output tile for the warp that owns TMEM lane quarter `quarter`: tcgen05.ld gives
// lane = row, register = column; a 32 x 32 block is transposed through a padded per-warp shared buffer so that every
// global store instruction writes contiguous 128-byte row segments.  Arrives on tempty_bar_addr once the warp's
// share of the accumulator is in registers.
__device__ __forceinline__ void tc_epilogue_tile(const TcArgs& args, uint32_t tmem_base, int acc, uint32_t tempty_bar_addr,
                                                 int quarter, float* stg, int m0, int n0, int bi, int ks, bool has_k,
                                                 int lane, int chunk0 = 0, int chunks = TC_BN / 32, float beta_override = -1.f) {
    const float beta = beta_override >= 0.f ? beta_override : args.beta;
    const int row_base = m0 + quarter * 32;
    float* out_base;
    int ldo;
    if (args.partial != nullptr) {
        out_base = args.partial + (static_cast<size_t>(bi) * args.k_splits + ks) * args.M * args.N;
        ldo = args.N;
    } else {
        out_base = args.C + bi * args.sC;
        ldo = args.ldc;
    }
    const int rows_valid = min(32, args.M - row_base);      // may be <= 0 for padding tiles
    const bool final_out = args.partial == nullptr;
    const bool vec = (ldo % 4 == 0) && ((reinterpret_cast<uintptr_t>(out_base) & 15) == 0) && (n0 + TC_BN <= args.N);
#pragma unroll 1
    for (int chunk = chunk0; chunk < chunk0 + chunks; ++chunk) {
        uint32_t v[32];
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) +
                               static_cast<uint32_t>(acc * TC_BN + chunk * 32);
        tmem_ld32(taddr, v);
        if (chunk == chunk0 + chunks - 1) {
            // the accumulator is in registers now: hand the TMEM buffer back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty_bar_addr);
        }
#pragma unroll
        for (int j = 0; j < 32; j += 4)          // lane = row; 16-byte chunk j/4 goes to slot (j/4) ^ (row & 7)
            *reinterpret_cast<float4*>(stg + lane * 32 + (((j >> 2) ^ (lane & 7)) << 2)) =
                has_k ? make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]),
                                    __uint_as_float(v[j + 3]))
                      : make_float4(0.f, 0.f, 0.f, 0.f);
        __syncwarp();
        if (vec) {
            // lane -> (row = 4*it + lane/8, float4 column = lane%8): 4 rows x 128 contiguous bytes per store
            const int c4 = (lane & 7) * 4, col = n0 + chunk * 32 + c4;
            float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (final_out && args.bias != nullptr) bias4 = *reinterpret_cast<const float4*>(args.bias + col);
            // beta != 0: fetch the 8 old values first -- interleaved with the stores the compiler must keep
            // each load behind the previous store (possible aliasing) and the epilogue becomes a chain of
            // eight global round trips per 32-column chunk
            float4 cold[8];
            const bool rmw = final_out && beta != 0.f;
            if (rmw) {
#pragma unroll
                for (int it = 0; it < 8; ++it) {
                    const int rr = 4 * it + (lane >> 3);
                    cold[it] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (rr < rows_valid)
                        cold[it] = *reinterpret_cast<const float4*>(out_base + static_cast<size_t>(row_base + rr) * ldo + col);
                }
            }
#pragma unroll
            for (int it = 0; it < 8; ++it) {
                const int rr = 4 * it + (lane >> 3);
                if (rr < rows_valid) {
                    float4 val = *reinterpret_cast<const float4*>(stg + rr * 32 + (((lane & 7) ^ (rr & 7)) << 2));
                    float4* p = reinterpret_cast<float4*>(out_base + static_cast<size_t>(row_base + rr) * ldo + col);
                    if (final_out) {
                        val.x = val.x * args.alpha + bias4.x; val.y = val.y * args.alpha + bias4.y;
                        val.z = val.z * args.alpha + bias4.z; val.w = val.w * args.alpha + bias4.w;
                        if (rmw) {
                            val.x += beta * cold[it].x; val.y += beta * cold[it].y;
                            val.z += beta * cold[it].z; val.w += beta * cold[it].w;
                        }
                    }
                    *p = val;
                }
            }
        } else {
            const int col = n0 + chunk * 32 + lane;
            if (col < args.N) {
                const float bias = (final_out && args.bias != nullptr) ? args.bias[col] : 0.f;
                for (int rr = 0; rr < rows_valid; ++rr) {
                    float val = stg[rr * 32 + ((((lane >> 2) ^ (rr & 7)) << 2) | (lane & 3))];
                    float* p = out_base + static_cast<size_t>(row_base + rr) * ldo + col;
                    if (final_out) {
                        val = val * args.alpha + bias;
                        if (beta != 0.f) val += beta * (*p);
                    }
                    *p = val;
                }
            }
        }
        __syncwarp();
    }
}

// BPRE: the B operand is a weight matrix that tc_presplit_b_kernel has already split and laid out as one
// ready-to-copy blob per (column tile, K block): a single bulk copy per stage replaces the B half of the
// producers' work, and the registers it frees double-buffer the A loads (two K blocks in flight per group).
constexpr uint32_t TC_B_BLOB_BYTES = 2 * TC_PART_BYTES;     // B_hi part, B_lo part

// APRE: the mirror image for the generated-operand weight gradient of the bilinear form (K = every pair): the small
// [rows, 128] operand is pre-split into blobs, the producers generate the wide operand (double-buffered).
// MNMAJ: both operands stored [K][MN] (C = A^T B) and fed to the tensor core MN-major (A_KCONTIG = B_KCONTIG = false).
template <bool A_KCONTIG, bool B_KCONTIG, int GROUPS, bool BPRE, bool APRE = false, bool MNMAJ = false>
__global__ void __launch_bounds__(tc_threads(GROUPS), 1) gemm_tc_kernel(const TcArgs args) {
    constexpr int TC_PRODUCER_WARPS = 4 * GROUPS, TC_MMA_WARP = 4 * GROUPS, TC_GROUPS = GROUPS;
    static_assert(GROUPS <= TC_STAGES, "a producer group may run at most one stage-round ahead of the MMA warp");
    // (no integer round trip on this pointer: the compiler must keep seeing shared memory, or every
    //  operand store degrades to a generic ST)
    extern __shared__ __align__(1024) uint8_t smem[];
    float* epi_stage = reinterpret_cast<float*>(smem + size_t(TC_STAGES) * TC_STAGE_BYTES);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + size_t(TC_STAGES) * TC_STAGE_BYTES + TC_EPI_BYTES);
    // bars: full[3], empty[3], tmem_full[2], tmem_empty[2], then the TMEM base address
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 10);
    const uint32_t bar0 = smem_u32(bars);
    auto full_bar = [&](int s) { return bar0 + 8u * s; };
    auto empty_bar = [&](int s) { return bar0 + 8u * (TC_STAGES + s); };
    auto tfull_bar = [&](int a) { return bar0 + 8u * (2 * TC_STAGES + a); };
    auto tempty_bar = [&](int a) { return bar0 + 8u * (2 * TC_STAGES + 2 + a); };

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int s = 0; s < TC_STAGES; ++s) {
            mbar_init(full_bar(s), (BPRE || APRE) ? 5 : 4);   // one arrive per producer warp (+ the expect_tx arrive of the blob)
            mbar_init(empty_bar(s), 1);   // tcgen05.commit
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(tfull_bar(a), 1);   // tcgen05.commit
            mbar_init(tempty_bar(a), 4);  // one arrive per epilogue warp
        }
        fence_barrier_init();
    }
    if (warp == TC_MMA_WARP) tmem_alloc(smem_u32(tmem_slot), TC_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int tiles_mn = args.tiles_m * args.tiles_n;
    const int total_tiles = tiles_mn * args.k_splits * args.batch;

    if (warp < TC_PRODUCER_WARPS) {
        // ===== producers: TC_GROUPS groups of 4 warps take K blocks round-robin; a group issues its loads
        // before it waits for its shared-memory stage, so TC_GROUPS blocks of global loads are in flight
        const bool a_vec = (args.lda % 4 == 0) && ((reinterpret_cast<uintptr_t>(args.A) & 15) == 0) && (args.sA % 4 == 0);
        const bool b_vec = (args.ldb % 4 == 0) && ((reinterpret_cast<uintptr_t>(args.B) & 15) == 0) && (args.sB % 4 == 0);
        const int group = warp >> 2, tid = threadIdx.x & 127;
        if (BPRE) {
            // (batch == 1, k_splits == 1)  flat sequence q of this CTA's K blocks; this group takes q = group (mod GROUPS)
            const int kblocks = args.kblocks;
            const int my_tiles = blockIdx.x < total_tiles ? (total_tiles - 1 - blockIdx.x) / static_cast<int>(gridDim.x) + 1 : 0;
            const int total_q = my_tiles * kblocks;
            auto fetch = [&](int q, float4 (&v)[8]) {
                const int tile = blockIdx.x + (q / kblocks) * gridDim.x, kb = q % kblocks;
                fetch_operand<A_KCONTIG>(args.A, args.lda, (tile / args.tiles_n) * TC_BM, args.M, kb * TC_BK, args.K, a_vec,
                                         tid, v);
            };
            auto commit = [&](int q, const float4 (&v)[8]) {
                const int stage = q % TC_STAGES;
                const uint32_t phase = (q / TC_STAGES) & 1;
                mbar_wait(empty_bar(stage), phase ^ 1);      // the MMAs that read this stage have retired
                uint8_t* stb = smem + size_t(stage) * TC_STAGE_BYTES;
                if (tid == 0) {
                    const int tile = blockIdx.x + (q / kblocks) * gridDim.x, kb = q % kblocks;
                    const uint8_t* blob = args.Bpre + (static_cast<size_t>(tile % args.tiles_n) * kblocks + kb) * TC_B_BLOB_BYTES;
                    mbar_arrive_expect_tx(full_bar(stage), TC_B_BLOB_BYTES);
                    bulk_copy_g2s(smem_u32(stb + 2 * TC_PART_BYTES), blob, TC_B_BLOB_BYTES, full_bar(stage));
                }
                float* st = reinterpret_cast<float*>(stb);
                store_operand<A_KCONTIG>(st, st + TC_PART_BYTES / 4, tid, v);
                fence_proxy_async();          // generic-proxy stores -> visible to the tensor core
                __syncwarp();
                if (lane == 0) mbar_arrive(full_bar(stage));
            };
            float4 va0[8], va1[8];
            int q = group;
            if (q < total_q) fetch(q, va0);
            while (q < total_q) {
                if (q + GROUPS < total_q) fetch(q + GROUPS, va1);
                commit(q, va0);
                q += GROUPS;
                if (q >= total_q) break;
                if (q + GROUPS < total_q) fetch(q + GROUPS, va0);
                commit(q, va1);
                q += GROUPS;
            }
        }
        if (APRE) {
            // (batch == 1)  work items t = blockIdx.x, + gridDim.x, ...; jbase = K blocks of the earlier items, so that the
            // stage / phase bookkeeping runs on across items exactly like the MMA warp's
            int jbase = 0;
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
                const int ks = t / tiles_mn, rem = t - ks * tiles_mn;
                const int mtile = rem / args.tiles_n, n0 = (rem % args.tiles_n) * TC_BN;
                const int kbeg = ks * args.k_per_split, kend = min(args.K, kbeg + args.k_per_split);
                const int total_q = kend > kbeg ? (kend - kbeg + TC_BK - 1) / TC_BK : 0;
                auto fetch = [&](int q, float4 (&v)[8]) {
                    if (args.bscale == nullptr) {
                        fetch_operand<B_KCONTIG>(args.B, args.ldb, n0, args.N, kbeg + q * TC_BK, kend, b_vec, tid, v);
                    } else {
                        // every column tile reads the same [K, 128] matrix, scaled per K row by this tile's weight
                        const int kq = kbeg + q * TC_BK, nt = n0 / TC_BN;
                        fetch_operand<B_KCONTIG>(args.B, args.ldb, 0, TC_BN, kq, kend, b_vec, tid, v);
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            int r, c;
                            tile_coord<B_KCONTIG>(tid, i, r, c);
                            const int k = kq + 4 * c;
                            const float* sp = args.bscale + static_cast<size_t>(k) * args.lds + nt;
                            v[i].x *= k < kend ? sp[0] : 0.f;
                            v[i].y *= k + 1 < kend ? sp[args.lds] : 0.f;
                            v[i].z *= k + 2 < kend ? sp[2 * static_cast<size_t>(args.lds)] : 0.f;
                            v[i].w *= k + 3 < kend ? sp[3 * static_cast<size_t>(args.lds)] : 0.f;
                        }
                    }
                };
                auto commit = [&](int q, const float4 (&v)[8]) {
                    const int j = jbase + q, stage = j % TC_STAGES;
                    const uint32_t phase = (j / TC_STAGES) & 1;
                    mbar_wait(empty_bar(stage), phase ^ 1);
                    uint8_t* stb = smem + size_t(stage) * TC_STAGE_BYTES;
                    if (tid == 0) {
                        const uint8_t* blob = args.Apre + (static_cast<size_t>(mtile) * args.kblocks + kbeg / TC_BK + q) * TC_B_BLOB_BYTES;
                        mbar_arrive_expect_tx(full_bar(stage), TC_B_BLOB_BYTES);
                        bulk_copy_g2s(smem_u32(stb), blob, TC_B_BLOB_BYTES, full_bar(stage));       // A_hi, A_lo parts
                    }
                    float* st = reinterpret_cast<float*>(stb);
                    store_operand<B_KCONTIG>(st + 2 * (TC_PART_BYTES / 4), st + 3 * (TC_PART_BYTES / 4), tid, v);
                    fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(full_bar(stage));
                };
                float4 vb0[8], vb1[8];
                int q = ((group - jbase) % GROUPS + GROUPS) % GROUPS;       // first K block of the item with (jbase + q) % GROUPS == group
                if (q < total_q) fetch(q, vb0);
                while (q < total_q) {
                    if (q + GROUPS < total_q) fetch(q + GROUPS, vb1);
                    commit(q, vb0);
                    q += GROUPS;
                    if (q >= total_q) break;
                    if (q + GROUPS < total_q) fetch(q + GROUPS, vb0);
                    commit(q, vb1);
                    q += GROUPS;
                }
                jbase += total_q;
            }
        }
        int j = 0;                                   // running K-block index of this CTA
        for (int t = blockIdx.x; !BPRE && !APRE && t < total_tiles; t += gridDim.x) {
            const int bi = t / (tiles_mn * args.k_splits), tb = t - bi * (tiles_mn * args.k_splits);
            const int ks = tb / tiles_mn, rem = tb - ks * tiles_mn;
            const int m0 = (rem / args.tiles_n) * TC_BM, n0 = (rem % args.tiles_n) * TC_BN;
            const int kbeg = ks * args.k_per_split;
            const int kend = min(args.K, kbeg + args.k_per_split);
            const float* Ab = args.A + bi * args.sA;
            const float* Bb = args.B + bi * args.sB;
            for (int k0 = kbeg; k0 < kend; k0 += TC_BK, ++j) {
                if ((j % TC_GROUPS) != group) continue;
                const int stage = j % TC_STAGES;
                const uint32_t phase = (j / TC_STAGES) & 1;
                float4 va[8], vb[8];
                if (MNMAJ) {
                    fetch_operand_mn(Ab, args.lda, m0, args.M, k0, kend, a_vec, tid, va);
                    fetch_operand_mn(Bb, args.ldb, n0, args.N, k0, kend, b_vec, tid, vb);
                } else {
                    fetch_operand<A_KCONTIG>(Ab, args.lda, m0, args.M, k0, kend, a_vec, tid, va);
                    fetch_operand<B_KCONTIG>(Bb, args.ldb, n0, args.N, k0, kend, b_vec, tid, vb);
                }
                mbar_wait(empty_bar(stage), phase ^ 1);      // the MMAs that read this stage have retired
                float* st = reinterpret_cast<float*>(smem + size_t(stage) * TC_STAGE_BYTES);
                if (MNMAJ) {
                    uint8_t* sb = smem + size_t(stage) * TC_STAGE_BYTES;
                    store_operand_mn(sb, sb + TC_MN_PART_BYTES, tid, va);
                    store_operand_mn(sb + 2 * TC_MN_PART_BYTES, sb + 3 * TC_MN_PART_BYTES, tid, vb);
                } else {
                    store_operand<A_KCONTIG>(st, st + TC_PART_BYTES / 4, tid, va);
                    store_operand<B_KCONTIG>(st + 2 * (TC_PART_BYTES / 4), st + 3 * (TC_PART_BYTES / 4), tid, vb);
                }
                fence_proxy_async();          // generic-proxy stores -> visible to the tensor core
                __syncwarp();
                if (lane == 0) mbar_arrive(full_bar(stage));
            }
        }
    } else if (warp == TC_MMA_WARP) {
        // ===== MMA issuer (one elected lane) =====
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
                const int ks = (t % (tiles_mn * args.k_splits)) / tiles_mn;
                const int kbeg = ks * args.k_per_split;
                const int kend = min(args.K, kbeg + args.k_per_split);
                mbar_wait(tempty_bar(acc), acc_phase ^ 1);     // epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * TC_BN);
                uint32_t accumulate = 0;
                for (int k0 = kbeg; k0 < kend; k0 += TC_BK) {
                    mbar_wait(full_bar(stage), phase);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(smem + size_t(stage) * TC_STAGE_BYTES);
                    if (MNMAJ) {
                        const uint32_t a_hi = sa, a_lo = sa + TC_MN_PART_BYTES;
                        const uint32_t b_hi = sa + 2 * TC_MN_PART_BYTES, b_lo = sa + 3 * TC_MN_PART_BYTES;
#pragma unroll
                        for (int kk = 0; kk < TC_BK / 8; ++kk) {
                            const uint32_t koff = kk * 8 * 128;          // eight k rows per MMA
                            umma_tf32(d_tmem, make_desc_mn(a_lo + koff), make_desc_mn(b_hi + koff), TC_IDESC_MN, accumulate);
                            umma_tf32(d_tmem, make_desc_mn(a_hi + koff), make_desc_mn(b_lo + koff), TC_IDESC_MN, 1u);
                            umma_tf32(d_tmem, make_desc_mn(a_hi + koff), make_desc_mn(b_hi + koff), TC_IDESC_MN, 1u);
                            accumulate = 1u;
                        }
                    } else {
                        const uint32_t a_hi = sa, a_lo = sa + TC_PART_BYTES;
                        const uint32_t b_hi = sa + 2 * TC_PART_BYTES, b_lo = sa + 3 * TC_PART_BYTES;
#pragma unroll
                        for (int kk = 0; kk < TC_BK / 8; ++kk) {
                            const uint32_t koff = kk * 2 * TC_PLANE_BYTES;   // two 16-byte K chunks per MMA
                            umma_tf32(d_tmem, make_desc(a_lo + koff), make_desc(b_hi + koff), TC_IDESC, accumulate);
                            umma_tf32(d_tmem, make_desc(a_hi + koff), make_desc(b_lo + koff), TC_IDESC, 1u);
                            umma_tf32(d_tmem, make_desc(a_hi + koff), make_desc(b_hi + koff), TC_IDESC, 1u);
                            accumulate = 1u;
                        }
                    }
                    umma_commit(empty_bar(stage));             // stage is free once these MMAs retire
                    if (++stage == TC_STAGES) { stage = 0; phase ^= 1; }
                }
                umma_commit(tfull_bar(acc));                   // accumulator complete
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
        __syncwarp();
    } else {
        // ===== epilogue: warps 17..20 own TMEM lane quarters (warp % 4) =====
        // tcgen05.ld gives lane = row, register = column.  A 32x32 block is transposed through a padded
        // per-warp shared buffer so that every global store instruction writes one contiguous 128-byte
        // row segment (lane = column) instead of 32 scattered 16-byte pieces.
        const int quarter = warp & 3;
        float* stg = epi_stage + quarter * TC_EPI_WARP_FLOATS;
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
            const int bi = t / (tiles_mn * args.k_splits), tb = t - bi * (tiles_mn * args.k_splits);
            const int ks = tb / tiles_mn, rem = tb - ks * tiles_mn;
            const int m0 = (rem / args.tiles_n) * TC_BM, n0 = (rem % args.tiles_n) * TC_BN;
            const bool has_k = ks * args.k_per_split < args.K;
            mbar_wait(tfull_bar(acc), acc_phase);
            tc_fence_after();
            tc_epilogue_tile(args, tmem_base, acc, tempty_bar(acc), quarter, stg, m0, n0, bi, ks, has_k, lane, 0, TC_BN / 32,
                             (args.seq_k && ks > 0) ? 1.f : -1.f);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == TC_MMA_WARP) tmem_dealloc(tmem_base, TC_TMEM_COLS);
}

// ---- K <= 128 projections with a weight operand, row operand resident in TENSOR MEMORY ----------------------
// x W with W = [128, H*128]: the H column tiles of a 128-row tile share the row operand, so it is split ONCE per row
// tile (128 rows x K <= 128, hi and lo) into TMEM columns 256..511 (tcgen05.st from the producers' registers,
// row = lane) and read by tcgen05.mma as the A operand, while the weight blobs stream through five 33 KB shared-memory
// stages by bulk copy.  The producers work once per H tiles instead of once per tile; what remains is MMA issue and the
// 64 KB-per-tile store.  Roles: warps 0-7 producers (TMEM lane quarter warp & 3, K half warp >> 2), warp 8 blob loader,
// warp 9 MMA issuer, warps 10-17 epilogue (two per TMEM lane quarter, a column half each).
// TMEM: accumulators [0,128) and [128,256), A_hi [256,384), A_lo [384,512).
constexpr int TA_PRODUCER_WARPS = 8, TA_LOADER_WARP = 8, TA_MMA_WARP = 9, TA_KB = 4;
constexpr int TA_BSTAGES = 5, TA_EPI_WARPS = 8, TA_THREADS = (10 + TA_EPI_WARPS) * 32;
constexpr size_t TA_EPI_BYTES = size_t(TA_EPI_WARPS) * TC_EPI_WARP_FLOATS * 4;
constexpr size_t TA_SMEM_BYTES = size_t(TA_BSTAGES) * TC_B_BLOB_BYTES + TA_EPI_BYTES + 768 + 256;
constexpr uint32_t TA_COL_AHI = 256, TA_COL_ALO = 384;

template <int MODE>      // 0: store the tiles, 1: row-dot epilogue, 2: row-accumulate epilogue
__global__ void __launch_bounds__(TA_THREADS, 1) gemm_tc_tmema_kernel(const TcArgs args) {
    constexpr bool ROWDOT = MODE == 1, ROWACC = MODE == 2;
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* b_stage = smem;                                           // [TA_BSTAGES][B_hi part, B_lo part]
    float* epi_stage = reinterpret_cast<float*>(b_stage + size_t(TA_BSTAGES) * TC_B_BLOB_BYTES);
    uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(epi_stage) + TA_EPI_BYTES);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 6 + 2 * TA_BSTAGES);
    const uint32_t bar0 = smem_u32(bars);
    const uint32_t a_full = bar0, a_empty = bar0 + 8;
    auto tfull_bar = [&](int a) { return bar0 + 8u * (2 + a); };
    auto tempty_bar = [&](int a) { return bar0 + 8u * (4 + a); };
    auto b_full = [&](int s) { return bar0 + 8u * (6 + s); };
    auto b_empty = [&](int s) { return bar0 + 8u * (6 + TA_BSTAGES + s); };
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        mbar_init(a_full, TA_PRODUCER_WARPS);
        mbar_init(a_empty, 1);
        for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), TA_EPI_WARPS); }
        for (int i = 0; i < TA_BSTAGES; ++i) { mbar_init(b_full(i), 1); mbar_init(b_empty(i), 1); }
        fence_barrier_init();
    }
    if (warp == TA_MMA_WARP) tmem_alloc(smem_u32(tmem_slot), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int kblocks = args.kblocks, tiles_n = args.tiles_n, tiles_m = args.tiles_m;

    if (warp < TA_PRODUCER_WARPS) {
        // warp -> TMEM lane quarter (warp & 3) and K half (warp >> 2); lane = row of the quarter
        const int quarter = warp & 3, khalf = warp >> 2;
        const bool a_vec = (args.lda % 4 == 0) && ((reinterpret_cast<uintptr_t>(args.A) & 15) == 0);
        int it = 0;
        for (int mi = blockIdx.x; mi < tiles_m; mi += gridDim.x, ++it) {
            const int row = mi * TC_BM + quarter * 32 + lane;
            const float* src = args.A + static_cast<size_t>(row) * args.lda;
            // The row's 64 values of this K half are loaded BEFORE the wait for the A region of tensor memory: the loads
            // of row tile i + 1 then fly while the MMAs of tile i still read tile i's operand (they used to be issued
            // after the wait, 16 at a time: four exposed HBM latencies per row tile).
            float4 av[16];
            const int kbase = khalf * 64;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int k = kbase + 4 * j;
                if (k >= kblocks * TC_BK) {
                    av[j] = make_float4(0.f, 0.f, 0.f, 0.f);           // columns beyond the K blocks in use are never read
                } else if (row < args.M && a_vec && k + 4 <= args.K) {
                    av[j] = *reinterpret_cast<const float4*>(src + k);
                } else {
                    float t[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) t[e] = (row < args.M && k + e < args.K) ? src[k + e] : 0.f;
                    av[j] = make_float4(t[0], t[1], t[2], t[3]);
                }
            }
            mbar_wait(a_empty, (it & 1) ^ 1);            // the MMAs of the previous row tile have retired
            tc_fence_after();
#pragma unroll
            for (int c16 = 0; c16 < 4; ++c16) {
                const int k0 = kbase + c16 * 16;
                if (k0 >= kblocks * TC_BK) break;
                uint32_t hi[16], lo[16];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 v = av[4 * c16 + j];
                    const float t[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const uint32_t h = __float_as_uint(t[e]) & 0xffffe000u;
                        hi[4 * j + e] = h;
                        lo[4 * j + e] = __float_as_uint(t[e] - __uint_as_float(h));
                    }
                }
                const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
                tmem_st16(lane_base + TA_COL_AHI + k0, hi);
                tmem_st16(lane_base + TA_COL_ALO + k0, lo);
            }
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(a_full);
        }
    } else if (warp == TA_LOADER_WARP) {
        if (lane == 0) {
            int q = 0;
            for (int mi = blockIdx.x; mi < tiles_m; mi += gridDim.x)
                for (int n = 0; n < tiles_n; ++n)
                    for (int kb = 0; kb < kblocks; ++kb, ++q) {
                        const int stage = q % TA_BSTAGES;
                        mbar_wait(b_empty(stage), ((q / TA_BSTAGES) & 1) ^ 1);
                        const uint8_t* blob = args.Bpre + (static_cast<size_t>(n) * kblocks + kb) * TC_B_BLOB_BYTES;
                        mbar_arrive_expect_tx(b_full(stage), TC_B_BLOB_BYTES);
                        bulk_copy_g2s(smem_u32(b_stage + size_t(stage) * TC_B_BLOB_BYTES), blob, TC_B_BLOB_BYTES, b_full(stage));
                    }
        }
        __syncwarp();
    } else if (warp == TA_MMA_WARP) {
        if (lane == 0) {
            int q = 0, acc = 0, it = 0;
            uint32_t acc_phase = 0;
            constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((TC_BN >> 3) << 17) | ((TC_BM >> 4) << 24);
            for (int mi = blockIdx.x; mi < tiles_m; mi += gridDim.x, ++it) {
                mbar_wait(a_full, it & 1);
                tc_fence_after();
                for (int n = 0; n < tiles_n; ++n) {
                    mbar_wait(tempty_bar(acc), acc_phase ^ 1);
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * TC_BN);
                    uint32_t accumulate = 0;
                    for (int kb = 0; kb < kblocks; ++kb, ++q) {
                        const int stage = q % TA_BSTAGES;
                        mbar_wait(b_full(stage), (q / TA_BSTAGES) & 1);
                        tc_fence_after();
                        const uint32_t b_hi = smem_u32(b_stage + size_t(stage) * TC_B_BLOB_BYTES), b_lo = b_hi + TC_PART_BYTES;
#pragma unroll
                        for (int kk = 0; kk < TC_BK / 8; ++kk) {
                            const uint32_t koff = kk * 2 * TC_PLANE_BYTES;
                            const uint32_t acol = static_cast<uint32_t>(kb * TC_BK + kk * 8);
                            umma_tf32_ts(d_tmem, tmem_base + TA_COL_ALO + acol, make_desc(b_hi + koff), IDESC, accumulate);
                            umma_tf32_ts(d_tmem, tmem_base + TA_COL_AHI + acol, make_desc(b_lo + koff), IDESC, 1u);
                            umma_tf32_ts(d_tmem, tmem_base + TA_COL_AHI + acol, make_desc(b_hi + koff), IDESC, 1u);
                            accumulate = 1u;
                        }
                        umma_commit(b_empty(stage));
                    }
                    umma_commit(tfull_bar(acc));
                    if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                }
                umma_commit(a_empty);                    // the resident operand may be replaced once these retire
            }
        }
        __syncwarp();
    } else {
        const int quarter = warp & 3, ew = warp - (TA_MMA_WARP + 1);
        constexpr int CH = (TC_BN / 32) / (TA_EPI_WARPS / 4);
        float* stg = epi_stage + ew * TC_EPI_WARP_FLOATS;
        int acc = 0;
        uint32_t acc_phase = 0;
        if (ROWDOT) {
            // bilinear-form epilogue: lane = row keeps the 64 values of rd_t[row] that face this warp's column half in
            // registers for all column tiles of the row tile; one scalar per (row, column tile, half) leaves the SM
            static_assert(CH == 2, "row-dot epilogue assumes two 32-column chunks per epilogue warp");
            const int half = ew / 4;
            for (int mi = blockIdx.x; mi < tiles_m; mi += gridDim.x) {
                const int row = mi * TC_BM + quarter * 32 + lane;
                float4 t[16];
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    t[j] = row < args.M ? *reinterpret_cast<const float4*>(args.rd_t + static_cast<size_t>(row) * 128 + half * 64 + 4 * j)
                                        : make_float4(0.f, 0.f, 0.f, 0.f);
                for (int n = 0; n < tiles_n; ++n) {
                    mbar_wait(tfull_bar(acc), acc_phase);
                    tc_fence_after();
                    float s = 0.f;
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        uint32_t v[32];
                        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) +
                                               static_cast<uint32_t>(acc * TC_BN + (half * 2 + c) * 32);
                        tmem_ld32(taddr, v);
                        if (c == 1) {           // the accumulator is in registers: hand the TMEM buffer back
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive(tempty_bar(acc));
                        }
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float4 tv = t[c * 8 + j];
                            s += __uint_as_float(v[4 * j]) * tv.x + __uint_as_float(v[4 * j + 1]) * tv.y +
                                 __uint_as_float(v[4 * j + 2]) * tv.z + __uint_as_float(v[4 * j + 3]) * tv.w;
                        }
                    }
                    if (row < args.M) args.rd_out[(static_cast<long long>(n) * 2 + half) * args.rd_ld + row] = s;
                    if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                }
            }
        } else if (ROWACC) {
            // weighted sum of the column tiles: lane = row keeps the 64 running sums of its column half in registers
            // over all column tiles of the row tile, and stores them once
            static_assert(CH == 2, "row-accumulate epilogue assumes two 32-column chunks per epilogue warp");
            const int half = ew / 4;
            for (int mi = blockIdx.x; mi < tiles_m; mi += gridDim.x) {
                const int row = mi * TC_BM + quarter * 32 + lane;
                const float* wrow = args.rd_t + static_cast<size_t>(row < args.M ? row : 0) * args.rd_ld;
                float4 sum[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) sum[j] = make_float4(0.f, 0.f, 0.f, 0.f);
                for (int n = 0; n < tiles_n; ++n) {
                    const float wgt = row < args.M ? wrow[n] : 0.f;
                    mbar_wait(tfull_bar(acc), acc_phase);
                    tc_fence_after();
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        uint32_t v[32];
                        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) +
                                               static_cast<uint32_t>(acc * TC_BN + (half * 2 + c) * 32);
                        tmem_ld32(taddr, v);
                        if (c == 1) {
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive(tempty_bar(acc));
                        }
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            float4& a4 = sum[c * 8 + j];
                            a4.x += wgt * __uint_as_float(v[4 * j]);     a4.y += wgt * __uint_as_float(v[4 * j + 1]);
                            a4.z += wgt * __uint_as_float(v[4 * j + 2]); a4.w += wgt * __uint_as_float(v[4 * j + 3]);
                        }
                    }
                    if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                }
                if (row < args.M) {
                    float* o = args.rd_out + static_cast<size_t>(row) * 128 + half * 64;
#pragma unroll
                    for (int j = 0; j < 16; ++j) *reinterpret_cast<float4*>(o + 4 * j) = sum[j];
                }
            }
        } else {
            for (int mi = blockIdx.x; mi < tiles_m; mi += gridDim.x)
                for (int n = 0; n < tiles_n; ++n) {
                    mbar_wait(tfull_bar(acc), acc_phase);
                    tc_fence_after();
                    tc_epilogue_tile(args, tmem_base, acc, tempty_bar(acc), quarter, stg, mi * TC_BM, n * TC_BN, 0, 0, true, lane,
                                     (ew / 4) * CH, CH);
                    if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == TA_MMA_WARP) tmem_dealloc(tmem_base, 512);
}

// One blob per (128-column tile nt, 32-wide K block kb) of the N x K operand op(B)^T: exactly the B_hi / B_lo half of
// a shared-memory stage (8 chunk planes of [128 rows][16 B] + pad each), so the GEMM moves it with one bulk copy.
__global__ void __launch_bounds__(256)
tc_presplit_b_kernel(const float* __restrict__ B, int ldb, int b_kcontig, int N, int K, int kblocks,
                     uint8_t* __restrict__ blobs) {
    const int blob = blockIdx.x, nt = blob / kblocks, kb = blob - nt * kblocks;
    const int n0 = nt * TC_BN, k0 = kb * TC_BK;
    float* hi = reinterpret_cast<float*>(blobs + static_cast<size_t>(blob) * TC_B_BLOB_BYTES);
    float* lo = hi + TC_PART_BYTES / 4;
    // (the four quarters of a blob are independent: gridDim.y = 4 blocks of one element each per thread, so that the
    //  launch -- tens of them per step sit on the critical path -- is one memory round trip long, not four)
    for (int idx = blockIdx.y * 256 + threadIdx.x; idx < TC_BN * (TC_BK / 4); idx += 256 * gridDim.y) {
        int r, c;
        if (b_kcontig) { c = idx & 7; r = idx >> 3; } else { r = idx & (TC_BN - 1); c = idx >> 7; }
        const int n = n0 + r, k = k0 + 4 * c;
        float t[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            t[q] = 0.f;
            if (n < N && k + q < K)
                t[q] = b_kcontig ? B[static_cast<size_t>(n) * ldb + k + q] : B[static_cast<size_t>(k + q) * ldb + n];
        }
        split_store(hi, lo, c, r, make_float4(t[0], t[1], t[2], t[3]));
    }
}

// bytes of the pre-split blob array of a [rows, <= 128] operand used as the short side of a weight-gradient GEMM
size_t gemm_presplit_bytes(int rows) {
    return static_cast<size_t>(ceil_div(rows < 0 ? 0 : rows, TC_BK)) * TC_B_BLOB_BYTES;
}

int launch_splitk_reduce(const float* partial, int splits, int M, int N, float alpha, float beta, float* C,
                         int ldc, const float* bias, cudaStream_t st, int batch, long long sC);

// returns 1 if the launch was taken by the tensor-core path, 0 if the caller should use the SIMT kernel
int launch_gemm_tc(int ta, int tb, int M, int N, int K, float alpha, const float* A, int lda, const float* B,
                   int ldb, float beta, float* C, int ldc, const float* bias, void* ws, size_t ws_bytes,
                   cudaStream_t st, int* taken, int batch, long long sA, long long sB, long long sC, void* pre_ws,
                   size_t pre_bytes, const float* bscale, int lds) {
    *taken = 0;
    if (K < 1 || batch < 1) return GCGCN_OK;
    if (static_cast<double>(M) * N * K * batch < 2.0e6) return GCGCN_OK;   // tiny: not worth a 128x128 tile
    TcArgs a;
    a.M = M; a.N = N; a.K = K; a.lda = lda; a.ldb = ldb; a.ldc = ldc;
    a.A = A; a.B = B; a.bias = bias; a.C = C; a.alpha = alpha; a.beta = beta;
    a.tiles_m = ceil_div(M, TC_BM);
    a.tiles_n = ceil_div(N, TC_BN);
    a.batch = batch; a.sA = sA; a.sB = sB; a.sC = sC;
    a.rd_t = nullptr; a.rd_out = nullptr; a.rd_ld = 0; a.bscale = bscale; a.lds = lds; a.seq_k = 0;
    const int tiles = a.tiles_m * a.tiles_n * batch;
    const int sms = sm_count();
    int splits = 1;
    if (tiles < sms && K >= 4096) {
        // one wave: as many K slices as fit the SMs without a second, partially filled wave
        splits = std::min(std::max(sms / tiles, 1), ceil_div(K, 512));
        const size_t per = static_cast<size_t>(M) * N * sizeof(float) * batch;
        if (ws == nullptr) splits = 1;
        else splits = static_cast<int>(std::min<size_t>(splits, ws_bytes / per));
        if (splits < 2) splits = 1;
    }
    a.k_per_split = K;
    a.partial = nullptr;
    if (splits > 1) {
        a.k_per_split = ceil_div(ceil_div(K, splits), TC_BK) * TC_BK;
        splits = ceil_div(K, a.k_per_split);
        a.partial = static_cast<float*>(ws);
    }
    a.k_splits = splits;
    int grid = std::min(sms, tiles * splits);
    // generated-operand weight gradient (K = every pair of the batch): one CTA per tile walks the K ranges in order and
    // adds each range's accumulator into C, so that no single tensor-core accumulation is longer than 4096 rows
    const bool seq = bscale != nullptr;
    if (seq) {
        a.k_per_split = 4096;
        a.k_splits = splits = ceil_div(K, a.k_per_split);
        const size_t per = static_cast<size_t>(M) * N * sizeof(float);
        if (splits > 1 && ws != nullptr && per * splits <= ws_bytes && (reinterpret_cast<uintptr_t>(ws) & 15) == 0) {
            // room for one partial per range: plain split-K over the ranges, every CTA takes (tile, range) items
            // round-robin (all SMs busy), the fp32 reduction adds them up
            a.partial = static_cast<float*>(ws);
            a.seq_k = 0;
            grid = std::min(sms, tiles * splits);
        } else {
            a.partial = nullptr;
            a.seq_k = splits > 1 ? 1 : 0;
            grid = std::min(sms, tiles);
        }
    }
    a.Bpre = nullptr;
    a.kblocks = ceil_div(K, TC_BK);
    // weight-like B operand (small, reused by every 128-row tile of a tall A): pre-split it once per call
    const size_t blob_total = static_cast<size_t>(a.tiles_n) * a.kblocks * TC_B_BLOB_BYTES;
    const bool bpre = batch == 1 && splits == 1 && !seq && !ta && M >= 4096 &&
                      static_cast<size_t>(N) * K * sizeof(float) <= (size_t(8) << 20) && ws != nullptr &&
                      blob_total <= ws_bytes && (reinterpret_cast<uintptr_t>(ws) & 15) == 0;
    if (bpre) {
        tc_presplit_b_kernel<<<dim3(a.tiles_n * a.kblocks, 4), 256, 0, st>>>(B, ldb, tb != 0, N, K, a.kblocks, static_cast<uint8_t*>(ws));
        GCGCN_CHECK_LAUNCH("gemm_presplit_b");
        a.Bpre = static_cast<const uint8_t*>(ws);
    }
    // generated-operand weight gradient: the short [rows, <= 256] operand (A, transposed) is pre-split into blobs that
    // every column tile re-uses.  The other weight gradients run MN-major: blobs only pay for themselves where the
    // wide operand has to be generated (measured on [119808 x 128]^T [119808 x N]: N = 256: 95 us with blobs, 66 us
    // MN-major; N = 1024: 230 us against 216 us).
    a.Apre = nullptr;
    const size_t ablob_total = static_cast<size_t>(a.tiles_m) * a.kblocks * TC_B_BLOB_BYTES;
    const bool apre = bscale != nullptr && !bpre && batch == 1 && ta && !tb && K >= 8192 && M <= 2 * TC_BM &&
                      a.tiles_n >= 2 && (seq ? (a.partial != nullptr || tiles <= sms) : tiles * splits <= sms) &&
                      pre_ws != nullptr && ablob_total <= pre_bytes && (reinterpret_cast<uintptr_t>(pre_ws) & 15) == 0;
    if (bscale != nullptr && !apre)
        return fail(GCGCN_ERR_UNSUPPORTED, "gemm: the generated-operand product needs the pre-split weight-gradient path "
                    "(A transposed, K >= 8192, M <= 256, N >= 256, a pre-split workspace)");
    if (apre) {
        tc_presplit_b_kernel<<<dim3(a.tiles_m * a.kblocks, 4), 256, 0, st>>>(A, lda, /*kcontig=*/0, M, K, a.kblocks,
                                                                  static_cast<uint8_t*>(pre_ws));
        GCGCN_CHECK_LAUNCH("gemm_presplit_a");
        a.Apre = static_cast<const uint8_t*>(pre_ws);
    }
    // op(A)[m,k]: stored [M][K] (K contiguous) when !ta, [K][M] when ta.
    // op(B)[k,n] as the N x K operand: stored [N][K] (K contiguous) when tb, [K][N] when !tb.
    const bool a_kc = !ta, b_kc = (tb != 0);
#define GCGCN_TC_LAUNCH(AK, BK, G, ...)                                                                                 \
    do {                                                                                                                \
        static std::atomic<unsigned long long> prepared{0};                                                             \
        GCGCN_TRY(set_smem_once(prepared, gemm_tc_kernel<AK, BK, G, __VA_ARGS__>, TC_SMEM_BYTES, "gemm_tc smem"));      \
        gemm_tc_kernel<AK, BK, G, __VA_ARGS__><<<grid, tc_threads(G), TC_SMEM_BYTES, st>>>(a);                          \
    } while (0)
    // K <= 128 with a pre-split weight operand: the row operand stays resident in tensor memory across the column tiles
    // (also for a single column tile: 40 us against 44 us for [119808,128]x[128,128])
    const bool tmema = bpre && a.kblocks <= TA_KB;
    if (tmema) {
        static std::atomic<unsigned long long> prepared{0};
        GCGCN_TRY(set_smem_once(prepared, gemm_tc_tmema_kernel<0>, TA_SMEM_BYTES, "gemm_tc_tmema smem"));
        gemm_tc_tmema_kernel<0><<<std::min(sms, a.tiles_m), TA_THREADS, TA_SMEM_BYTES, st>>>(a);
    } else if (apre) GCGCN_TC_LAUNCH(false, false, 2, false, true);
    else if (bpre) GCGCN_TC_LAUNCH(true, true, 3, true);
    else if (a_kc && b_kc) GCGCN_TC_LAUNCH(true, true, 3, false);
    else if (a_kc && !b_kc) GCGCN_TC_LAUNCH(true, false, 3, false);
    else if (!a_kc && b_kc) GCGCN_TC_LAUNCH(false, true, 3, false);
    // (never more producer groups than stages: a group two stage-rounds ahead would pass its parity wait on the
    //  empty barrier one phase early and overwrite a stage the MMA warp has not consumed -- 4 groups hang)
    else GCGCN_TC_LAUNCH(false, false, 3, false, false, true);
#undef GCGCN_TC_LAUNCH
    timing_set_work(2.0 * M * N * K * batch);
    GCGCN_CHECK_LAUNCH(tmema ? "gemm_tc_nn<A in TMEM>"
                             : apre ? "gemm_tc_tn<presplit A>"
                             : bpre ? (tb ? "gemm_tc_nt<presplit B>" : "gemm_tc_nn<presplit B>")
                             : ta ? (tb ? "gemm_tc_tt" : "gemm_tc_tn<MN-major>") : (tb ? "gemm_tc_nt" : "gemm_tc_nn"));
    if (splits > 1 && a.partial != nullptr)
        GCGCN_TRY(launch_splitk_reduce(a.partial, splits, M, N, alpha, beta, C, ldc, bias, st, batch, sC));
    *taken = 1;
    return GCGCN_OK;
}

// Row-dot / row-accumulate GEMMs over a [M, K <= 128] row operand that stays resident in tensor memory per row tile
// (split hi/lo) while B [K, N] (N a multiple of 128) streams through shared memory as pre-split blobs; the accumulator
// tiles are consumed from TMEM and never stored:
//   mode 1  part[(nt * 2 + half) * ld + m] = sum_{c in half of tile nt} (A B)[m][128 nt + c] T[m][c]
//           -- the bilinear form out[p, r] = sum_b (h W')[p, r*128 + b] t[p, b]
//   mode 2  out[m][c] = sum_nt T[m * ld + nt] (A B)[m][128 nt + c]
//           -- its input gradients, dt[p, b] = sum_r dout[p, r] (h W')[p, r*128 + b]
int launch_gemm_rowop(int mode, int M, int N, int K, const float* A, int lda, const float* B, int ldb, const float* T,
                      float* out, long long ld, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (M <= 0 || N <= 0) return GCGCN_OK;
    if (K < 1 || K > TA_KB * TC_BK || N % TC_BN != 0)
        return fail(GCGCN_ERR_UNSUPPORTED, "gemm_rowop: needs 1 <= K <= %d and N a multiple of %d (K %d, N %d)", TA_KB * TC_BK,
                    TC_BN, K, N);
    TcArgs a;
    a.M = M; a.N = N; a.K = K; a.lda = lda; a.ldb = ldb; a.ldc = 0;
    a.A = A; a.B = B; a.bias = nullptr; a.C = nullptr; a.partial = nullptr; a.alpha = 1.f; a.beta = 0.f;
    a.tiles_m = ceil_div(M, TC_BM); a.tiles_n = N / TC_BN; a.k_splits = 1; a.k_per_split = K;
    a.kblocks = ceil_div(K, TC_BK); a.batch = 1; a.sA = a.sB = a.sC = 0; a.Apre = nullptr;
    a.rd_t = T; a.rd_out = out; a.rd_ld = ld; a.bscale = nullptr; a.lds = 0; a.seq_k = 0;
    const size_t blob_total = static_cast<size_t>(a.tiles_n) * a.kblocks * TC_B_BLOB_BYTES;
    if (ws == nullptr || blob_total > ws_bytes || (reinterpret_cast<uintptr_t>(ws) & 15) != 0)
        return fail(GCGCN_ERR_WORKSPACE, "gemm_rowop: workspace of %zu bytes needed for the pre-split weights", blob_total);
    tc_presplit_b_kernel<<<dim3(a.tiles_n * a.kblocks, 4), 256, 0, st>>>(B, ldb, 0, N, K, a.kblocks, static_cast<uint8_t*>(ws));
    GCGCN_CHECK_LAUNCH("gemm_presplit_b");
    a.Bpre = static_cast<const uint8_t*>(ws);
    const int grid = std::min(sm_count(), a.tiles_m);
    if (mode == 1) {
        static std::atomic<unsigned long long> prepared{0};
        GCGCN_TRY(set_smem_once(prepared, gemm_tc_tmema_kernel<1>, TA_SMEM_BYTES, "gemm_tc_rowdot smem"));
        gemm_tc_tmema_kernel<1><<<grid, TA_THREADS, TA_SMEM_BYTES, st>>>(a);
    } else {
        static std::atomic<unsigned long long> prepared{0};
        GCGCN_TRY(set_smem_once(prepared, gemm_tc_tmema_kernel<2>, TA_SMEM_BYTES, "gemm_tc_rowacc smem"));
        gemm_tc_tmema_kernel<2><<<grid, TA_THREADS, TA_SMEM_BYTES, st>>>(a);
    }
    timing_set_work(2.0 * M * N * K);
    GCGCN_CHECK_LAUNCH(mode == 1 ? "gemm_tc_rowdot<A in TMEM>" : "gemm_tc_rowacc<A in TMEM>");
    return GCGCN_OK;
}

}  // namespace gcgcn
