// MAGGC graph block on the 5th-generation tensor cores: documents packed into 128-row tiles (sm_100a).
//
// The per-document block kernels (gcn_block.cu) give every (document, head) its own CTA and run the small products
// as mma.sync fragments: with DocRED's ~20 entities per document most of a 16-row fragment tile is padding and the
// kernel is bound by shared-memory fragment traffic.  Here consecutive documents are packed into tiles of <= 96 node
// rows (gcgcn_batch.tile_doc, built by the host) and two persistent CTAs per SM walk (tile, head) items:
//
//   S   = q_h q_h^T                     tcgen05.mma 128x96x16, both operands from shared memory       -> TMEM [0,96)
//   P   = block-diagonal softmax(S)     one thread per (row, half of the columns); entries outside the row's
//                                       document are exact zeros, so the packed product below is the per-document one
//                                       P is written to HBM (saved for backward) and, split hi/lo, back into TMEM
//   N_l = P Z_l                         tcgen05.mma 128x64x96, A = P from TENSOR MEMORY, B = Z_l^T planes in smem
//   g_l = relu((E_l + N_l) / r) ; F_l = g_l + x_l                                      (G:106-113, G:47-49)
//   Z_1 = Zx_1 + g_0 Winner_1           tcgen05.mma 128x64x64, A = g_0 planes, B = pre-split weight blob
//
// All products are 3xTF32 (hi/lo operand split, fp32 accumulate in TMEM; see gemm_tc.cu).  Configuration: the GloVe
// model's MAGGC block (two sub-layers of 64 columns, 8 heads of width 16) and its 4-head variant of the entity sweep
// (head width 32), eval mode; everything else takes the per-document kernels.  Results match them to fp32 rounding (different summation order in the softmax and the MMAs).
#include "common.cuh"
#include "mma_tf32.cuh"
#include "tc_ptx.cuh"

#include <cstdlib>

namespace gcgcn {

constexpr int TL_THREADS = 256;
constexpr int TL_GD = 64;                        // sub-layer width (two sub-layers); head width DH = 16 or 32 is a template parameter
constexpr int TL_ROWS = GCGCN_TILE_ROWS;         // node rows per tile = K extent of P Z
static_assert(TL_ROWS == 96, "thread mapping and TMEM layout below assume 96-row tiles");
constexpr int TL_HALF = TL_ROWS / 2;             // attention columns per thread
// Operand layouts in shared memory
//   K-major, no swizzle (row operands written one row per thread): [K/4 planes][rows][16 B] (+16 B per plane so that a
//     warp writing 32 rows x 16 B per plane and a quarter warp writing 8 planes of one row are both conflict-free)
//   MN-major, 128-byte swizzle with 32-byte base (the only MN-major layout the tensor core takes for 32-bit operands;
//     used for the Z_l tiles, which arrive row-major [k = node row][n = column] and are written by coalesced 16-byte
//     accesses): two column blocks of [96 k][32 n] fp32, rows 128 B apart, the 32-byte chunk index XORed with (k % 4)
//     -- the canonical UMMA "Major-MN / SWIZZLE_128B_BASE32B" atom, 4 k x 128 B
constexpr int TL_PLANE_M = TL_ROWS * 16 + 16;
constexpr int TL_PLANE_N = 64 * 16 + 16;
template <int DH>
constexpr int TL_Q_PART_OF = (DH / 4) * TL_PLANE_M;      // q_h  [96 rows][DH k]   K-major
constexpr int TL_ZBLK = TL_ROWS * 128;                   // one [96 k][32 n] column block of Z_l
constexpr int TL_B_PART = 2 * TL_ZBLK;                   // Z_l              [96 k][64 n]      MN-major SW128
constexpr int TL_G_PART = (TL_GD / 4) * TL_PLANE_M;      // g_0              [96 rows][64 k]   K-major (aliases the Z region)
constexpr int TL_W_PART = (TL_GD / 4) * TL_PLANE_N;      // Winner_1^T       [64 n][64 k]      K-major
constexpr int TL_ZG_BYTES = ((2 * (TL_G_PART > TL_B_PART ? TL_G_PART : TL_B_PART)) + 1023) / 1024 * 1024;
constexpr int TL_STAGE_LD = 64 * 4 + 16;                 // staging row: 64 fp32 + 16 B (conflict-free row-per-lane 16 B stores)
constexpr int TL_STAGE_BYTES = TL_ROWS * TL_STAGE_LD;    // accumulator tiles on their way from TMEM to coalesced stores
static_assert(2 * TL_Q_PART_OF<32> <= TL_STAGE_BYTES, "the q planes live in the staging buffer until S is done");
constexpr int TL_OFF_ZG = 0;                             // 1024-aligned (swizzle atoms)
constexpr int TL_OFF_WHI = TL_OFF_ZG + TL_ZG_BYTES, TL_OFF_WLO = TL_OFF_WHI + TL_W_PART;
constexpr int TL_OFF_STAGE = TL_OFF_WLO + TL_W_PART;
constexpr int TL_OFF_XCH = TL_OFF_STAGE + TL_STAGE_BYTES;   // [3][2][128] floats: cross-half max / sum exchanges
constexpr int TL_OFF_BAR = TL_OFF_XCH + 3 * 256 * 4;
constexpr int TL_SMEM_BYTES = TL_OFF_BAR + 64 + 1024 /*align*/;
static_assert(2 * (TL_SMEM_BYTES + 1024) <= 227 * 1024, "two CTAs per SM");
constexpr int TL_WBLOB_BYTES = 2 * TL_W_PART;            // per head, hi then lo
// TMEM columns: S, overwritten in place by P hi; P lo; one 64-column accumulator (N_0, then g_0 Winner, then N_1).
// 256 columns, so two CTAs share an SM's tensor memory.
constexpr uint32_t TL_COL_PHI = 0, TL_COL_PLO = TL_ROWS, TL_COL_ACC = 2 * TL_ROWS, TL_TMEM_COLS = 256;
static_assert(TL_COL_ACC + TL_GD <= TL_TMEM_COLS, "TMEM budget");
// kind::tf32, fp32 accumulate, M = 128 (the MMA always spans 128 TMEM lanes; lanes >= 96 are unused: a row of D
// depends on its own row of A only, so whatever the A operand reads there never reaches a real row).  BMN: B is MN-major.
template <int N, bool BMN>
constexpr uint32_t TL_IDESC = (1u << 4) | (2u << 7) | (2u << 10) | (BMN ? (1u << 16) : 0u) | ((uint32_t(N) >> 3) << 17) |
                              ((128u >> 4) << 24);

__device__ __forceinline__ uint64_t tl_desc(uint32_t smem_addr, uint32_t lbo) {      // K-major, no swizzle
    uint64_t d = (smem_addr >> 4) & 0x3FFFu;
    d |= static_cast<uint64_t>(lbo >> 4) << 16;          // leading (K) byte offset: one chunk plane
    d |= static_cast<uint64_t>(128 >> 4) << 32;          // stride (M/N) byte offset: one 8-row core matrix
    d |= static_cast<uint64_t>(1) << 46;
    return d;
}
__device__ __forceinline__ uint64_t tl_desc_mn(uint32_t smem_addr) {                 // MN-major, SWIZZLE_128B_BASE32B
    uint64_t d = (smem_addr >> 4) & 0x3FFFu;
    d |= static_cast<uint64_t>(TL_ZBLK >> 4) << 16;      // leading byte offset: the next 32-column block
    d |= static_cast<uint64_t>(512 >> 4) << 32;          // stride byte offset: the next atom of 4 k rows
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(1) << 61;                 // SWIZZLE_128B_BASE32B
    return d;
}
__device__ __forceinline__ void tl_split(float x, float& hi, float& lo) {
    hi = __uint_as_float(__float_as_uint(x) & 0xffffe000u);
    lo = x - hi;
}
__device__ __forceinline__ void tl_split4(const float4 v, float4& hi, float4& lo) {
    tl_split(v.x, hi.x, lo.x); tl_split(v.y, hi.y, lo.y); tl_split(v.z, hi.z, lo.z); tl_split(v.w, hi.w, lo.w);
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void sts4(uint32_t addr, const float4 v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float4 lds4(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
    return v;
}
// byte offset of (k row, 16-byte chunk c16 of the 64 columns) inside one hi/lo part of the swizzled Z tile
__device__ __forceinline__ uint32_t tl_zoff(int row, int c16) {
    const int c = c16 & 7;
    return static_cast<uint32_t>((c16 >> 3) * TL_ZBLK + row * 128 + (((((c >> 1) ^ (row & 3)) << 1) | (c & 1)) << 4));
}

// Winner_1 of every head as a ready-to-copy B operand: out[h][hi|lo][k / 4][n][k % 4], B(n, k) = W_{h,1}[k][n]
__global__ void __launch_bounds__(256)
tile_wprep_kernel(const float* __restrict__ Winner, int layers, uint8_t* __restrict__ out) {
    const int h = blockIdx.x;
    const float* W = Winner + (static_cast<size_t>(h) * layers + 1) * D * TL_GD;
    uint8_t* o = out + static_cast<size_t>(h) * TL_WBLOB_BYTES;
    for (int idx = threadIdx.x; idx < TL_GD * TL_GD; idx += blockDim.x) {
        const int k = idx / TL_GD, n = idx - k * TL_GD;
        float hi, lo;
        tl_split(W[idx], hi, lo);
        const int off = (k >> 2) * TL_PLANE_N + n * 16 + (k & 3) * 4;
        *reinterpret_cast<float*>(o + off) = hi;
        *reinterpret_cast<float*>(o + TL_W_PART + off) = lo;
    }
}

struct TileFwdArgs {
    const int* tile_doc;
    const int* node_ptr;
    const long long* pair_ptr;
    const int* row_doc;
    const float* q;
    float* P;
    float* Z;
    const float* E;
    const uint8_t* Wblob;
    const float* x;
    float* G;
    float* F;
    int heads, num_tiles;
    long long total_pairs;
    float scale;
};

// Two thread mappings:
//   row mapping (TMEM side): warp w owns TMEM lane quarter w % 4 (rows 32 (w % 4) .. + 32 of the tile) and column half
//     w / 4; the two warps of quarter 3 (rows 96..127 do not exist) idle in these phases;
//   coalesced mapping (HBM side): thread t handles the 16-byte chunk t % 16 of rows t / 16 + 16 i, i < 6 -- a warp
//     touches two whole 256-byte row segments per instruction.  (With one row per lane every 16-byte global access of
//     a warp hit 32 different lines and the L1 data pipe, not HBM, bounded the kernel: ncu, profiles/r02_tile_fwd.md.)
// Accumulator tiles cross from the first mapping to the second through the staging buffer.
template <int DH>
__global__ void __launch_bounds__(TL_THREADS, 2) tile_fwd_kernel(const TileFwdArgs a) {
    constexpr int TL_Q_PART = TL_Q_PART_OF<DH>, QV = DH / 8;      // QV float4 of q per thread (half of the head slice)
    extern __shared__ uint8_t smem_raw[];
    const uint32_t sraw = smem_u32(smem_raw);
    const uint32_t sbase = (sraw + 1023u) & ~1023u;
    uint8_t* smem = smem_raw + (sbase - sraw);
    float* xch = reinterpret_cast<float*>(smem + TL_OFF_XCH);
    const uint32_t bar = sbase + TL_OFF_BAR;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + TL_OFF_BAR + 16);
    const uint32_t s_zg = sbase + TL_OFF_ZG, s_stage = sbase + TL_OFF_STAGE;
    const uint32_t s_qhi = s_stage, s_qlo = s_stage + TL_Q_PART;

    const int tid = threadIdx.x, warp = tid >> 5;
    const int r = tid & 127, half = tid >> 7;             // row mapping
    const bool rowthread = r < TL_ROWS;
    const int crow = tid >> 4, c16 = tid & 15;            // coalesced mapping
    if (tid == 0) {
        mbar_init(bar, 1);
        fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(smem_u32(tmem_slot), TL_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(r & ~31) << 16);   // this warp's lane quarter

    const int HD = a.heads * D;
    const int items = a.num_tiles * a.heads;
    uint32_t phase = 0;
    int cur_h = -1;
    // The first phase's operands are fetched one item ahead (tile geometry at the top of the previous item, q rows
    // before its last wait), so an item starts with its data in registers instead of three dependent round trips to
    // L2/HBM.  (Fetching the Zx_0 tile ahead as well was measured slower: 24 more live registers spill.)
    int n_row0 = 0, n_rows = 0;
    float4 n_q[QV];
    auto fetch_geometry = [&](int item) {
        if (item < items) {
            const int tile = item % a.num_tiles;
            const int d0 = a.tile_doc[tile], d1 = a.tile_doc[tile + 1];
            n_row0 = a.node_ptr[d0];
            n_rows = a.node_ptr[d1] - n_row0;
        }
    };
    auto fetch_operands = [&](int item) {
        const int h = item / a.num_tiles;
#pragma unroll
        for (int i = 0; i < QV; ++i) n_q[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (item < items && rowthread && r < n_rows) {
            const float* qp = a.q + static_cast<size_t>(n_row0 + r) * D + h * DH + half * (DH / 2);
#pragma unroll
            for (int i = 0; i < QV; ++i) n_q[i] = ld4g(qp + 4 * i);
        }
    };
    fetch_geometry(blockIdx.x);
    fetch_operands(blockIdx.x);
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
        const int h = item / a.num_tiles;
        const int row0 = n_row0, rows = n_rows;
        const bool rv = r < rows;                          // rows <= TL_ROWS
        // coalesced mapping: element offset of (row crow + 16 i, chunk c16) in the [rows, H*128] slabs / in x
        const size_t cslab = static_cast<size_t>(row0 + crow) * HD + h * D + c16 * 4;      // + i * 16 * HD + l * 64
        const size_t cx = static_cast<size_t>(row0 + crow) * D + c16 * 4;                  // + i * 16 * D + l * 64

        // ---- stage q_h (A and B operand of S) and, when the head changes, its dense-connect weights ----
        if (rowthread) {
            const uint32_t dst = (QV * half) * TL_PLANE_M + r * 16;
#pragma unroll
            for (int i = 0; i < QV; ++i) {
                float4 hi, lo;
                tl_split4(n_q[i], hi, lo);
                sts4(s_qhi + dst + i * TL_PLANE_M, hi);
                sts4(s_qlo + dst + i * TL_PLANE_M, lo);
            }
        }
        fetch_geometry(item + gridDim.x);
        if (h != cur_h) {
            const float4* src = reinterpret_cast<const float4*>(a.Wblob + static_cast<size_t>(h) * TL_WBLOB_BYTES);
            for (int i = tid; i < TL_WBLOB_BYTES / 16; i += TL_THREADS) sts4(sbase + TL_OFF_WHI + i * 16, __ldg(src + i));
            cur_h = h;
        }
        fence_proxy_async();
        tc_fence_before();             // orders the previous item's tcgen05.ld before the MMAs issued below
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            constexpr uint32_t IDESC = TL_IDESC<TL_ROWS, false>;
#pragma unroll
            for (int kk = 0; kk < DH / 8; ++kk) {
                const uint32_t koff = kk * 2 * TL_PLANE_M;
                const uint64_t dh = tl_desc(s_qhi + koff, TL_PLANE_M);
                const uint64_t dl = tl_desc(s_qlo + koff, TL_PLANE_M);
                umma_tf32(tmem_base + TL_COL_PHI, dl, dh, IDESC, kk > 0 ? 1u : 0u);
                umma_tf32(tmem_base + TL_COL_PHI, dh, dl, IDESC, 1u);
                umma_tf32(tmem_base + TL_COL_PHI, dh, dh, IDESC, 1u);
            }
            umma_commit(bar);
        }
        // ---- meanwhile: the Zx_0 tile -> swizzled MN-major planes, and this row's document range ----
        {
            float4 z[6];
#pragma unroll
            for (int i = 0; i < 6; ++i)
                z[i] = crow + 16 * i < rows ? ld4g(a.Z + cslab + static_cast<size_t>(i) * 16 * HD) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int i = 0; i < 6; ++i) {
                float4 hi, lo;
                tl_split4(z[i], hi, lo);
                const uint32_t off = tl_zoff(crow + 16 * i, c16);
                sts4(s_zg + off, hi);
                sts4(s_zg + TL_B_PART + off, lo);
            }
        }
        int lo_col = 0, hi_col = 0;
        long long prow = 0;
        if (rv) {
            const int b = a.row_doc[row0 + r];
            const int n0 = a.node_ptr[b], n1 = a.node_ptr[b + 1];
            lo_col = n0 - row0;
            hi_col = n1 - row0;
            prow = static_cast<long long>(h) * a.total_pairs + a.pair_ptr[b] +
                   static_cast<long long>(r - lo_col) * (n1 - n0) - lo_col;           // + tile column j
        }
        // ---- softmax over the row's document columns (G:137-139); P saved, P hi/lo -> TMEM ----
        mbar_wait(bar, phase);
        phase ^= 1;
        tc_fence_after();
        // Three passes over the row's 48 scores, 16 at a time straight from tensor memory (re-reading TMEM and taking
        // the exponential twice is cheaper than keeping 48 values live: at 128 registers per thread they spilled).
        const int jb = half * TL_HALF;
        const uint32_t srow = lane_addr + TL_COL_PHI + jb;
        float m = -INFINITY;
        if (rowthread) {
#pragma unroll
            for (int c0 = 0; c0 < TL_HALF; c0 += 16) {
                uint32_t s[16];
                tmem_ld16(srow + c0, s);
                tmem_ld_wait();
#pragma unroll
                for (int c = 0; c < 16; ++c) {
                    const int j = jb + c0 + c;
                    if (j >= lo_col && j < hi_col) m = fmaxf(m, __uint_as_float(s[c]));
                }
            }
            xch[half * 128 + r] = m;
        }
        __syncthreads();
        float zsum = 0.f;
        float mk = 0.f;                // max * scale * log2(e): e = exp2(s * k - mk)
        const float kexp = a.scale * 1.4426950408889634f;
        if (rowthread) {
            m = fmaxf(xch[r], xch[128 + r]);
            mk = m * kexp;
#pragma unroll
            for (int c0 = 0; c0 < TL_HALF; c0 += 16) {
                uint32_t s[16];
                tmem_ld16(srow + c0, s);
                tmem_ld_wait();
#pragma unroll
                for (int c = 0; c < 16; ++c) {
                    const int j = jb + c0 + c;
                    if (j >= lo_col && j < hi_col) zsum += exp2f(fmaf(__uint_as_float(s[c]), kexp, -mk));
                }
            }
            xch[256 + half * 128 + r] = zsum;
        }
        __syncthreads();
        if (rowthread) {
            zsum = xch[256 + r] + xch[256 + 128 + r];
            const float inv = rv ? 1.0f / zsum : 0.f;
            float psum = 0.f;
#pragma unroll
            for (int c0 = 0; c0 < TL_HALF; c0 += 16) {
                uint32_t s[16], lo[16];
                tmem_ld16(srow + c0, s);
                tmem_ld_wait();
#pragma unroll
                for (int c = 0; c < 16; ++c) {
                    const int j = jb + c0 + c;
                    float p = 0.f;
                    if (j >= lo_col && j < hi_col) {
                        p = exp2f(fmaf(__uint_as_float(s[c]), kexp, -mk)) * inv;
                        a.P[prow + j] = p;
                    }
                    psum += p;
                    float ph, pl;
                    tl_split(p, ph, pl);
                    s[c] = __float_as_uint(ph);
                    lo[c] = __float_as_uint(pl);
                }
                tmem_st16(srow + c0, s);                                   // P hi over S, in place
                tmem_st16(lane_addr + TL_COL_PLO + jb + c0, lo);
            }
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            xch[512 + half * 128 + r] = psum;          // row sums of P (G:47-48); the reciprocal is taken where it is used
        }
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();

#pragma unroll
        for (int l = 0; l < 2; ++l) {
            // ---- N_l = P Z_l ----
            if (tid == 0) {
                tc_fence_after();
                constexpr uint32_t IDESC = TL_IDESC<TL_GD, true>;
#pragma unroll
                for (int kk = 0; kk < TL_ROWS / 8; ++kk) {
                    const uint64_t bh = tl_desc_mn(s_zg + kk * 1024);
                    const uint64_t bl = tl_desc_mn(s_zg + TL_B_PART + kk * 1024);
                    umma_tf32_ts(tmem_base + TL_COL_ACC, tmem_base + TL_COL_PLO + 8 * kk, bh, IDESC, kk > 0 ? 1u : 0u);
                    umma_tf32_ts(tmem_base + TL_COL_ACC, tmem_base + TL_COL_PHI + 8 * kk, bl, IDESC, 1u);
                    umma_tf32_ts(tmem_base + TL_COL_ACC, tmem_base + TL_COL_PHI + 8 * kk, bh, IDESC, 1u);
                }
                umma_commit(bar);
            }
            // the epilogue's HBM operands while the tensor core works
            float4 e4[6], x4[6];
#pragma unroll
            for (int i = 0; i < 6; ++i) {
                const bool ok = crow + 16 * i < rows;
                e4[i] = ok ? ld4g(a.E + cslab + static_cast<size_t>(i) * 16 * HD + l * TL_GD) : make_float4(0.f, 0.f, 0.f, 0.f);
                x4[i] = ok ? ld4g(a.x + cx + static_cast<size_t>(i) * 16 * D + l * TL_GD) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            if (l == 1) fetch_operands(item + gridDim.x);      // the next item's q rows
            mbar_wait(bar, phase);
            phase ^= 1;
            tc_fence_after();
            if (rowthread) {           // accumulator rows -> staging buffer
                uint32_t acc[32];
                tmem_ld32(lane_addr + TL_COL_ACC + half * 32, acc);
                const uint32_t dst = s_stage + r * TL_STAGE_LD + half * 128;
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    sts4(dst + 16 * i, make_float4(__uint_as_float(acc[4 * i]), __uint_as_float(acc[4 * i + 1]),
                                                   __uint_as_float(acc[4 * i + 2]), __uint_as_float(acc[4 * i + 3])));
            }
            tc_fence_before();
            __syncthreads();
            // g_l = relu((E_l + N_l) / r) ; F_l = g_l + x_l   (coalesced)
#pragma unroll
            for (int i = 0; i < 6; ++i) {
                const int row = crow + 16 * i;
                const float sum = xch[512 + row] + xch[512 + 128 + row];
                const float rinv = 1.0f / (sum + (sum == 0.f ? 1.f : 0.f));
                const float4 nv = lds4(s_stage + row * TL_STAGE_LD + c16 * 16);
                float4 g;
                g.x = fmaxf((e4[i].x + nv.x) * rinv, 0.f);
                g.y = fmaxf((e4[i].y + nv.y) * rinv, 0.f);
                g.z = fmaxf((e4[i].z + nv.z) * rinv, 0.f);
                g.w = fmaxf((e4[i].w + nv.w) * rinv, 0.f);
                if (row < rows) {
                    const size_t off = cslab + static_cast<size_t>(i) * 16 * HD + l * TL_GD;
                    *reinterpret_cast<float4*>(a.G + off) = g;
                    *reinterpret_cast<float4*>(a.F + off) = make_float4(g.x + x4[i].x, g.y + x4[i].y, g.z + x4[i].z, g.w + x4[i].w);
                }
                if (l == 0) {          // g_0 -> K-major A-operand planes of the dense-connect product (over the dead Z_0 tile)
                    float4 hi, lo;
                    tl_split4(g, hi, lo);
                    const uint32_t dst = s_zg + c16 * TL_PLANE_M + row * 16;
                    sts4(dst, hi);
                    sts4(dst + TL_G_PART, lo);
                }
            }
            if (l == 0) {
                // ---- Z_1 = Zx_1 + g_0 Winner_1 (G:103-105) ----
                fence_proxy_async();
                __syncthreads();
                if (tid == 0) {
                    tc_fence_after();
                    constexpr uint32_t IDESC = TL_IDESC<TL_GD, false>;
#pragma unroll
                    for (int kk = 0; kk < TL_GD / 8; ++kk) {
                        const uint64_t ah = tl_desc(s_zg + kk * 2 * TL_PLANE_M, TL_PLANE_M);
                        const uint64_t al = tl_desc(s_zg + TL_G_PART + kk * 2 * TL_PLANE_M, TL_PLANE_M);
                        const uint64_t bh = tl_desc(sbase + TL_OFF_WHI + kk * 2 * TL_PLANE_N, TL_PLANE_N);
                        const uint64_t bl = tl_desc(sbase + TL_OFF_WLO + kk * 2 * TL_PLANE_N, TL_PLANE_N);
                        umma_tf32(tmem_base + TL_COL_ACC, al, bh, IDESC, kk > 0 ? 1u : 0u);
                        umma_tf32(tmem_base + TL_COL_ACC, ah, bl, IDESC, 1u);
                        umma_tf32(tmem_base + TL_COL_ACC, ah, bh, IDESC, 1u);
                    }
                    umma_commit(bar);
                }
                float4 z[6];
#pragma unroll
                for (int i = 0; i < 6; ++i)
                    z[i] = crow + 16 * i < rows ? ld4g(a.Z + cslab + static_cast<size_t>(i) * 16 * HD + TL_GD)
                                                : make_float4(0.f, 0.f, 0.f, 0.f);
                mbar_wait(bar, phase);
                phase ^= 1;
                tc_fence_after();
                if (rowthread) {
                    uint32_t acc[32];
                    tmem_ld32(lane_addr + TL_COL_ACC + half * 32, acc);
                    const uint32_t dst = s_stage + r * TL_STAGE_LD + half * 128;
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        sts4(dst + 16 * i, make_float4(__uint_as_float(acc[4 * i]), __uint_as_float(acc[4 * i + 1]),
                                                       __uint_as_float(acc[4 * i + 2]), __uint_as_float(acc[4 * i + 3])));
                }
                tc_fence_before();
                __syncthreads();
#pragma unroll
                for (int i = 0; i < 6; ++i) {
                    const int row = crow + 16 * i;
                    const float4 nv = lds4(s_stage + row * TL_STAGE_LD + c16 * 16);
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (row < rows) {
                        v = make_float4(z[i].x + nv.x, z[i].y + nv.y, z[i].z + nv.z, z[i].w + nv.w);
                        *reinterpret_cast<float4*>(a.Z + cslab + static_cast<size_t>(i) * 16 * HD + TL_GD) = v;   // final Z_1, saved for backward
                    }
                    float4 hi, lo;
                    tl_split4(v, hi, lo);
                    const uint32_t off = tl_zoff(row, c16);
                    sts4(s_zg + off, hi);
                    sts4(s_zg + TL_B_PART + off, lo);
                }
                fence_proxy_async();
                __syncthreads();
            }
        }
        __syncthreads();               // the staging buffer is the next item's q planes
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, TL_TMEM_COLS);
}

static std::atomic<int>& tile_flag() {
    static std::atomic<int> on{[] {
        const char* e = std::getenv("GCGCN_TILE_BLOCKS");
        return (e != nullptr && e[0] == '0') ? 0 : 1;         // on unless GCGCN_TILE_BLOCKS=0
    }()};
    return on;
}
bool tile_blocks_enabled() { return tile_flag().load(std::memory_order_relaxed) != 0; }
bool set_tile_blocks(bool on) { return tile_flag().exchange(on ? 1 : 0) != 0; }

size_t tile_wblob_bytes(int heads) { return static_cast<size_t>(heads) * TL_WBLOB_BYTES; }

// MHA attention + MAGGC block forward on packed 128-row tiles.  Preconditions (checked by the caller): two sub-layers,
// head width 16 or 32, no dropout, bt->tile_doc present.
int launch_tile_fwd(const gcgcn_batch* bt, int heads, int layers, const float* q, float* P, float* Z, const float* E,
                    const float* Winner_rowmajor, const float* x, float* G, float* F, void* wblob_ws, cudaStream_t st) {
    if (bt->num_tiles <= 0) return GCGCN_OK;
    if (bt->tile_rows != TL_ROWS) return fail(GCGCN_ERR_INVALID_ARG, "tile_fwd: batch packed for %d-row tiles, kernel built for %d", bt->tile_rows, TL_ROWS);
    uint8_t* blob = static_cast<uint8_t*>(wblob_ws);
    tile_wprep_kernel<<<heads, 256, 0, st>>>(Winner_rowmajor, layers, blob);
    GCGCN_CHECK_LAUNCH("tile_wprep");
    static std::atomic<unsigned long long> prepared16{0}, prepared32{0};
    GCGCN_TRY(set_smem_once(prepared16, tile_fwd_kernel<16>, TL_SMEM_BYTES, "tile_fwd"));
    GCGCN_TRY(set_smem_once(prepared32, tile_fwd_kernel<32>, TL_SMEM_BYTES, "tile_fwd"));
    TileFwdArgs a;
    a.tile_doc = bt->tile_doc;
    a.node_ptr = bt->node_ptr;
    a.pair_ptr = reinterpret_cast<const long long*>(bt->pair_ptr);
    a.row_doc = bt->row_doc;
    a.q = q; a.P = P; a.Z = Z; a.E = E; a.Wblob = blob; a.x = x; a.G = G; a.F = F;
    a.heads = heads;
    a.num_tiles = bt->num_tiles;
    a.total_pairs = bt->total_pairs;
    const int dh = D / heads;
    a.scale = 1.0f / sqrtf(static_cast<float>(dh));
    const int items = bt->num_tiles * heads;
    const int grid = items < 2 * sm_count() ? items : 2 * sm_count();
    if (dh == 16) tile_fwd_kernel<16><<<grid, TL_THREADS, TL_SMEM_BYTES, st>>>(a);
    else if (dh == 32) tile_fwd_kernel<32><<<grid, TL_THREADS, TL_SMEM_BYTES, st>>>(a);
    else return fail(GCGCN_ERR_UNSUPPORTED, "tile_fwd: head width %d", dh);
    GCGCN_CHECK_LAUNCH("tile_fwd");
    return GCGCN_OK;
}

}  // namespace gcgcn
