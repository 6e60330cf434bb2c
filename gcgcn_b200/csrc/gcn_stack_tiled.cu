// Dense-connected GraphConv stack for graphs of up to 256 entities with sub-layer width 32 or 64 that the block
// kernels of gcn_block.cu do not take: the 128 / 256-entity sweep (BASELINE.json configs[3]), keep masks passed
// in as tensors, and a GraphConv used on its own.  One CTA per (document, head, 32-row tile) and one launch per
// sub-layer.
//
// Same contract and math as gcn_stack.cu (G:36-50 inside G:67-76 / G:103-113).  That kernel gives one CTA a
// whole (document, head): at n = 256 it owns 220 KB of shared memory, so one CTA of eight warps per SM walks
// load -> barrier -> product -> barrier phases with nothing to overlap them, and a batch offers only
// documents x heads CTAs (44 for the one-head CAGGC block of the 256-entity point).  Here the rows of the
// n x n attention map are cut into 32-row tiles:
//   forward, launch l:   G_l[tile] = relu((E_l + A[tile,:] Z_l) / r),  F_l[tile],  then the row-local dense
//                        connection  Z_{l+1}[tile] = Zx_{l+1}[tile] + g_{<=l}[tile] Winner_{l+1}
//   backward, launch "rows" l:  dN_l[tile] (= dE_l), dr, and  dA[tile,:] (+)= dN_l[tile] Z_l^T
//   backward, launch "cols" l:  dZ_l[tile] = A[:,tile]^T dN_l,  then the row-local push-down into dZ slabs m < l
// The cross-row dependencies (every row tile needs all rows of Z_l, every column tile all rows of dN_l) are
// carried by the kernel boundaries; each CTA keeps one [n, g] operand (<= 74 KB) and one 32-row tile
// (<= 33 KB) in shared memory, so two CTAs share an SM and 4-8x more of them are in flight.
// All products run on the tensor cores (mma.sync m16n8k8 TF32, 3xTF32 split of mma_tf32.cuh: fp32 parity).
#include "common.cuh"
#include "mma_tf32.cuh"

namespace gcgcn {

constexpr int TL_THREADS = 256;
constexpr int TL_WARPS = TL_THREADS / WARP;
constexpr int TL_ROWS = 32;     // rows of the attention map per CTA

template <int GD>
struct TileCfg {
    static constexpr int LDZ = GD + 8;      // [k][n] operands (B fragments): stride == 8 (mod 32)
    static constexpr int LDB = GD + 4;      // [m][k] / [n][k] operands (A and B^T fragments): stride == 4 (mod 8)
    static constexpr int NT = GD / 32;      // 8-column tiles per warp: 2 row tiles x 4 column groups of GD / 4
    static constexpr int CG = GD / 4;       // float4 column groups of a slab
};

__device__ __forceinline__ float4 tl_ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
// 16-byte global -> shared copies that do not pass through registers: a CTA issues all loads of its operand tiles
// back to back and waits once (the scalar load -> store loops exposed one L2 round trip per unrolled batch)
__device__ __forceinline__ void tl_cp16(float* smem_dst, const float* gsrc) {
    const uint32_t d = static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst));
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void tl_cp_wait_all() {
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ void tl_zero4(float* p) { *reinterpret_cast<float4*>(p) = make_float4(0.f, 0.f, 0.f, 0.f); }

// all rows [0, rows) of one sub-layer slab (GD columns at `src`, row stride HD) -> dst[rows_pad][ld], zero padded
template <int GD>
__device__ __forceinline__ void load_slab_rows(float* dst, int ld, const float* __restrict__ src, int HD, int rows,
                                               int rows_pad) {
    constexpr int CG = GD / 4;
    for (int idx = threadIdx.x; idx < rows_pad * CG; idx += TL_THREADS) {
        const int i = idx / CG, c4 = (idx - i * CG) * 4;
        if (i < rows) tl_cp16(dst + i * ld + c4, src + static_cast<size_t>(i) * HD + c4);
        else tl_zero4(dst + i * ld + c4);
    }
}

// rows [row0, row0 + 32) x columns [0, k8) of the document's n x n map -> As[32][lda], zero outside the document.
// vec: n % 4 == 0 and the map starts on a 16-byte boundary.
__device__ __forceinline__ void load_att_rows(float* As, int lda, const float* __restrict__ Ab, int n, int k8, int row0,
                                              bool vec) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int ii = warp; ii < TL_ROWS; ii += TL_WARPS) {
        const bool row_ok = row0 + ii < n;
        const float* src = Ab + static_cast<size_t>(row0 + ii) * n;
        float* dst = As + ii * lda;
        if (vec) {
            for (int c4 = lane * 4; c4 < k8; c4 += 4 * WARP) {
                if (row_ok && c4 < n) tl_cp16(dst + c4, src + c4);
                else tl_zero4(dst + c4);
            }
        } else {
            for (int j = lane; j < k8; j += WARP) dst[j] = (row_ok && j < n) ? src[j] : 0.f;
        }
    }
}

// C[16 x 8 NT] += A^T-stored product: A(m, k) = pa[k * lda + m] (the attention tile as it lies in memory, rows = k),
// B(k, n) = pb[k * ldb + n]; 3xTF32 like warp_gemm.  lda == 8 (mod 32) keeps the A fragment loads conflict-free.
template <int NT>
__device__ __forceinline__ void warp_gemm_at(float (&c)[NT][4], int ksteps, const float* __restrict__ pa, int lda,
                                             const float* __restrict__ pb, int ldb) {
    const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    const float* a0 = pa + t * lda + g;
    const float* b0 = pb + t * ldb + g;
#pragma unroll 2
    for (int ks = 0; ks < ksteps; ++ks) {
        uint32_t ah[4], al[4];
        split_tf32(a0[0], ah[0], al[0]);
        split_tf32(a0[8], ah[1], al[1]);
        split_tf32(a0[4 * lda], ah[2], al[2]);
        split_tf32(a0[4 * lda + 8], ah[3], al[3]);
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            uint32_t bh[2], bl[2];
            split_tf32(b0[nt * 8], bh[0], bl[0]);
            split_tf32(b0[nt * 8 + 4 * ldb], bh[1], bl[1]);
            mma_tf32(c[nt], al, bh);
            mma_tf32(c[nt], ah, bl);
            mma_tf32(c[nt], ah, bh);
        }
        a0 += 8 * lda;
        b0 += 8 * ldb;
    }
}

// ---------------------------------------------------------------------------------------------------
// forward, sub-layer l
template <int GD>
__global__ void __launch_bounds__(TL_THREADS, 2)
stack_tile_fwd_kernel(const int* __restrict__ node_ptr, const long long* __restrict__ pair_ptr,
                      const float* __restrict__ A, float* __restrict__ Z, const float* __restrict__ E,
                      const float* __restrict__ Winner, const float* __restrict__ keep, const float* __restrict__ x,
                      float* __restrict__ G, float* __restrict__ F, int l, int layers, int heads, int flags,
                      long long total_pairs) {
    using C = TileCfg<GD>;
    extern __shared__ __align__(16) float smem[];
    const int b = blockIdx.z, h = blockIdx.y, row0 = blockIdx.x * TL_ROWS;
    const int node0 = node_ptr[b];
    const int n = node_ptr[b + 1] - node0;
    if (row0 >= n) return;
    const int S = layers * GD, HD = heads * S;
    const int k8 = (n + 7) & ~7, lda = k8 + 4;
    const int kin = (l + 1) * GD, ldg = kin + 4;            // dense-connect inputs of sub-layer l + 1
    const int tile_floats = max(TL_ROWS * lda, TL_ROWS * (S + 4));

    float* Zl = smem;                                       // [k8][LDZ]   Z_l, all rows of the document
    float* As = Zl + static_cast<size_t>(k8) * C::LDZ;      // [32][lda]   attention rows of the tile; later g_{<=l}
    float* rs = As + tile_floats;                           // [32]        row normalisers

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const float* Ab = A + static_cast<long long>(h) * total_pairs + pair_ptr[b];
    const size_t colbase = static_cast<size_t>(h) * S + l * GD;
    const bool relu = flags & GCGCN_STACK_RELU, resid = flags & GCGCN_STACK_RESIDUAL;

    const long long abase = static_cast<long long>(h) * total_pairs + pair_ptr[b];
    const bool vec = (n & 3) == 0 && (abase & 3) == 0;
    load_slab_rows<GD>(Zl, C::LDZ, Z + static_cast<size_t>(node0) * HD + colbase, HD, n, k8);
    load_att_rows(As, lda, Ab, n, k8, row0, vec);
    tl_cp_wait_all();
    __syncthreads();
    for (int ii = warp; ii < TL_ROWS; ii += TL_WARPS) {     // r_i = rowsum + [rowsum == 0]   (G:47-49)
        float s = 0.f;
        for (int j = lane; j < k8; j += WARP) s += As[ii * lda + j];
        s = warp_sum(s);
        if (lane == 0) rs[ii] = s + (s == 0.f ? 1.f : 0.f);
    }
    __syncthreads();

    // out = (E + A Z_l) / r : warp (mt, ng) owns rows 16 mt .. + 15 and columns ng GD/4 .. + GD/4 - 1
    const int mt = warp >> 2, ng = warp & 3;
    float c[C::NT][4];
    zero_frag<C::NT>(c);
    warp_gemm<C::NT, false>(c, k8 / 8, As + (16 * mt) * lda, lda, Zl + 8 * C::NT * ng, C::LDZ);
    float2 o[2][C::NT];
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int ii = 16 * mt + g + 8 * half, i = row0 + ii;
        const float r = rs[ii];
#pragma unroll
        for (int nt = 0; nt < C::NT; ++nt) {
            o[half][nt] = make_float2(0.f, 0.f);
            if (i >= n) continue;
            const int cw = 8 * C::NT * ng + 8 * nt + 2 * t;
            const size_t off = static_cast<size_t>(node0 + i) * HD + colbase + cw;
            const float2 e2 = ld2g(E + off);
            float2 v;
            v.x = (e2.x + c[nt][2 * half]) / r;
            v.y = (e2.y + c[nt][2 * half + 1]) / r;
            if (relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); }
            *reinterpret_cast<float2*>(G + off) = v;
            o[half][nt] = v;
            float2 f = v;
            if (keep != nullptr) { const float2 k2 = ld2g(keep + off); f.x *= k2.x; f.y *= k2.y; }
            if (resid) {
                const float2 x2 = ld2g(x + static_cast<size_t>(node0 + i) * S + l * GD + cw);
                f.x += x2.x; f.y += x2.y;
            }
            *reinterpret_cast<float2*>(F + off) = f;
        }
    }
    if (l + 1 >= layers) return;

    // dense connection of the next sub-layer for the rows of this tile (row-local, G:72-73):
    //   Z_{l+1}[tile] = Zx_{l+1}[tile] + [g_0 .. g_l][tile] Winner_{l+1}[0 : (l+1) GD]
    __syncthreads();                                        // every warp is done with the attention rows
    float* Gt = As;                                         // [32][ldg]
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int ii = 16 * mt + g + 8 * half;
#pragma unroll
        for (int nt = 0; nt < C::NT; ++nt) {
            const int cw = 8 * C::NT * ng + 8 * nt + 2 * t;
            *reinterpret_cast<float2*>(Gt + ii * ldg + l * GD + cw) = o[half][nt];
        }
    }
    for (int idx = tid; idx < TL_ROWS * l * C::CG; idx += TL_THREADS) {     // g_m, m < l, from earlier launches
        const int ii = idx / (l * C::CG), c4 = (idx - ii * (l * C::CG)) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (row0 + ii < n) v = tl_ld4(G + static_cast<size_t>(node0 + row0 + ii) * HD + static_cast<size_t>(h) * S + c4);
        *reinterpret_cast<float4*>(Gt + ii * ldg + c4) = v;
    }
    __syncthreads();
    const size_t nextbase = static_cast<size_t>(h) * S + (l + 1) * GD;
    const float* wsrc = Winner + (static_cast<size_t>(h) * layers + (l + 1)) * S * GD;
#pragma unroll
    for (int nt = 0; nt < C::NT; ++nt)
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int i = row0 + 16 * mt + g + 8 * half;
            float2 v = make_float2(0.f, 0.f);
            if (i < n) v = ld2g(Z + static_cast<size_t>(node0 + i) * HD + nextbase + 8 * C::NT * ng + 8 * nt + 2 * t);
            c[nt][2 * half] = v.x;
            c[nt][2 * half + 1] = v.y;
        }
    warp_gemm<C::NT, false>(c, kin / 8, Gt + (16 * mt) * ldg, ldg, wsrc + 8 * C::NT * ng, GD);
#pragma unroll
    for (int nt = 0; nt < C::NT; ++nt)
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int i = row0 + 16 * mt + g + 8 * half;
            if (i >= n) continue;
            *reinterpret_cast<float2*>(Z + static_cast<size_t>(node0 + i) * HD + nextbase + 8 * C::NT * ng + 8 * nt + 2 * t) =
                make_float2(c[nt][2 * half], c[nt][2 * half + 1]);
        }
}

// ---------------------------------------------------------------------------------------------------
// backward "rows", sub-layer l: dN_l (= dE_l) and dr for the rows of the tile, dA[tile, :] (+)= dN_l Z_l^T
template <int GD>
__global__ void __launch_bounds__(TL_THREADS, 2)
stack_tile_bwd_rows_kernel(const int* __restrict__ node_ptr, const long long* __restrict__ pair_ptr,
                           const float* __restrict__ A, const float* __restrict__ Z, const float* __restrict__ G,
                           const float* __restrict__ keep, const float* __restrict__ dF,
                           const float* __restrict__ dZ, float* __restrict__ dE, float* __restrict__ dA, int l,
                           int layers, int heads, int flags, long long total_pairs) {
    using C = TileCfg<GD>;
    extern __shared__ __align__(16) float smem[];
    constexpr int TR = 64;      // rows per CTA here: the [n, g] operand is the only large tile, so 64 rows still leave
                                // room for two CTAs per SM and halve the per-row cost of loading it
    const int b = blockIdx.z, h = blockIdx.y, row0 = blockIdx.x * TR;
    const int node0 = node_ptr[b];
    const int n = node_ptr[b + 1] - node0;
    if (row0 >= n) return;
    const int S = layers * GD, HD = heads * S;
    const int n64 = (n + 63) & ~63;

    float* Ts = smem;                                        // [n64][LDB]  Z_l, all rows (B^T operand)
    float* dNs = Ts + static_cast<size_t>(n64) * C::LDB;     // [64][LDB]   dN_l of the tile
    float* rs = dNs + TR * C::LDB;                           // [64]
    float* drs = rs + TR;                                    // [64]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const long long abase = static_cast<long long>(h) * total_pairs + pair_ptr[b];
    const float* Ab = A + abase;
    float* dAb = dA + abase;
    const size_t colbase = static_cast<size_t>(h) * S + l * GD;
    const bool relu = flags & GCGCN_STACK_RELU;

    load_slab_rows<GD>(Ts, C::LDB, Z + static_cast<size_t>(node0) * HD + colbase, HD, n, n64);
    // (a), loads: everything the row-local phase needs from global memory is requested now, while the Z_l tile is
    // still in flight -- dG_l (dF, keep, what the sub-layers above pushed down), g_l, and at l == 0 the dr shares of
    // the sub-layers above (their dN = dE and g are final).  CG threads per row, NI rows per thread.
    constexpr int RPP = TL_THREADS / C::CG, NI = TR / RPP;
    const int cg = tid % C::CG, rg = tid / C::CG, c0 = cg * 4;
    float4 dgv[NI], g4v[NI];
    float upper[NI];
#pragma unroll
    for (int u = 0; u < NI; ++u) {
        const int i = row0 + rg + u * RPP;
        dgv[u] = g4v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        upper[u] = 0.f;
        if (i >= n) continue;
        const size_t off = static_cast<size_t>(node0 + i) * HD + colbase + c0;
        float4 dg = tl_ld4(dF + off);
        if (keep != nullptr) {
            const float4 k4 = tl_ld4(keep + off);
            dg.x *= k4.x; dg.y *= k4.y; dg.z *= k4.z; dg.w *= k4.w;
        }
        if (l < layers - 1) {
            const float4 s4 = tl_ld4(dZ + off);
            dg.x += s4.x; dg.y += s4.y; dg.z += s4.z; dg.w += s4.w;
        }
        dgv[u] = dg;
        g4v[u] = tl_ld4(G + off);
        if (l == 0) {
            for (int m = 1; m < layers; ++m) {
                const size_t om = static_cast<size_t>(node0 + i) * HD + static_cast<size_t>(h) * S + m * GD + c0;
                const float4 dm = tl_ld4(dE + om), gm = tl_ld4(G + om);
                upper[u] -= dm.x * gm.x + dm.y * gm.y + dm.z * gm.z + dm.w * gm.w;
            }
        }
    }
    const bool vec = (n & 3) == 0 && (abase & 3) == 0;
    for (int ii = warp; ii < TR; ii += TL_WARPS) {           // row normalisers straight from global memory
        float s = 0.f;
        if (row0 + ii < n) {
            const float* arow = Ab + static_cast<size_t>(row0 + ii) * n;
            if (vec) {
                for (int j = lane * 4; j < n; j += 4 * WARP) {
                    const float4 v = tl_ld4(arow + j);
                    s += (v.x + v.y) + (v.z + v.w);
                }
            } else {
                for (int j = lane; j < n; j += WARP) s += arow[j];
            }
        }
        s = warp_sum(s);
        if (lane == 0) { rs[ii] = s + (s == 0.f ? 1.f : 0.f); drs[ii] = 0.f; }
    }
    tl_cp_wait_all();
    __syncthreads();

    // (a), arithmetic: dOut = relu'(g) dG ; dN_l = dOut / r (shared + dE) ; dr = -sum_c dN g
#pragma unroll
    for (int u = 0; u < NI; ++u) {
        const int ii = rg + u * RPP, i = row0 + ii;
        float4 dn = make_float4(0.f, 0.f, 0.f, 0.f);
        float drp = 0.f;
        if (i < n) {
            float4 dg = dgv[u];
            const float4 g4 = g4v[u];
            if (relu) {
                dg.x = g4.x > 0.f ? dg.x : 0.f; dg.y = g4.y > 0.f ? dg.y : 0.f;
                dg.z = g4.z > 0.f ? dg.z : 0.f; dg.w = g4.w > 0.f ? dg.w : 0.f;
            }
            const float r = rs[ii];
            dn.x = dg.x / r; dn.y = dg.y / r; dn.z = dg.z / r; dn.w = dg.w / r;
            *reinterpret_cast<float4*>(dE + static_cast<size_t>(node0 + i) * HD + colbase + c0) = dn;
            drp = upper[u] - (dn.x * g4.x + dn.y * g4.y + dn.z * g4.z + dn.w * g4.w);
        }
        *reinterpret_cast<float4*>(dNs + ii * C::LDB + c0) = dn;
#pragma unroll
        for (int s = C::CG / 2; s > 0; s >>= 1) drp += __shfl_xor_sync(0xffffffffu, drp, s);
        if (cg == 0) drs[ii] = drp;
    }
    __syncthreads();

    // (c) dA[tile, :] (+)= dN_l Z_l^T (+ dr at l == 0), 64 columns per trip: warp (mt, ng) owns rows 16 mt .. + 15
    //     and columns 32 ng .. + 31 of the trip.  The values to accumulate onto are fetched before the product.
    const int mt = warp & 3, ng = warp >> 2;
    const bool accumulate = l != layers - 1;
    const bool pair_ok = (n & 1) == 0 && (abase & 1) == 0;       // (j, j + 1) pairs are 8-byte aligned
    for (int jp = 0; jp < n64; jp += 64) {
        float2 cur[2][4];
#pragma unroll
        for (int half = 0; half < 2; ++half)
#pragma unroll
            for (int nt = 0; nt < 4; ++nt) {
                cur[half][nt] = make_float2(0.f, 0.f);
                const int i = row0 + 16 * mt + g + 8 * half, j = jp + 32 * ng + 8 * nt + 2 * t;
                if (!accumulate || i >= n || j >= n) continue;
                const float* p = dAb + static_cast<size_t>(i) * n + j;
                if (pair_ok) cur[half][nt] = *reinterpret_cast<const float2*>(p);
                else { cur[half][nt].x = p[0]; if (j + 1 < n) cur[half][nt].y = p[1]; }
            }
        float c[4][4];
        zero_frag<4>(c);
        warp_gemm<4, true>(c, GD / 8, dNs + (16 * mt) * C::LDB, C::LDB, Ts + (jp + 32 * ng) * C::LDB, C::LDB);
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int ii = 16 * mt + g + 8 * half, i = row0 + ii;
            if (i >= n) continue;
            const float dr = (l == 0) ? drs[ii] : 0.f;
#pragma unroll
            for (int nt = 0; nt < 4; ++nt) {
                const int j = jp + 32 * ng + 8 * nt + 2 * t;
                if (j >= n) continue;
                float* p = dAb + static_cast<size_t>(i) * n + j;
                const float2 v = make_float2(c[nt][2 * half] + dr + cur[half][nt].x,
                                             c[nt][2 * half + 1] + dr + cur[half][nt].y);
                if (pair_ok) *reinterpret_cast<float2*>(p) = v;
                else { p[0] = v.x; if (j + 1 < n) p[1] = v.y; }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// backward "cols", sub-layer l: dZ_l[tile] = A[:, tile]^T dN_l, then the dense-connect push-down of those rows
template <int GD>
__global__ void __launch_bounds__(TL_THREADS, 2)
stack_tile_bwd_cols_kernel(const int* __restrict__ node_ptr, const long long* __restrict__ pair_ptr,
                           const float* __restrict__ A, const float* __restrict__ Winner,
                           const float* __restrict__ dE, float* __restrict__ dZ, int l, int layers, int heads,
                           long long total_pairs) {
    using C = TileCfg<GD>;
    extern __shared__ __align__(16) float smem[];
    const int b = blockIdx.z, h = blockIdx.y, j0 = blockIdx.x * TL_ROWS;
    const int node0 = node_ptr[b];
    const int n = node_ptr[b + 1] - node0;
    if (j0 >= n) return;
    const int S = layers * GD, HD = heads * S;
    const int k8 = (n + 7) & ~7;
    constexpr int LDU = TL_ROWS + 8;                         // == 8 (mod 32): conflict-free transposed-A fragments

    float* dNs = smem;                                       // [k8][LDZ]   dN_l, all rows (B operand)
    float* AsU = dNs + static_cast<size_t>(k8) * C::LDZ;     // [k8][LDU]   AsU[i][jj] = A[i][j0 + jj], as it lies in memory

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const long long abase = static_cast<long long>(h) * total_pairs + pair_ptr[b];
    const float* Ab = A + abase;
    const size_t colbase = static_cast<size_t>(h) * S + l * GD;
    const bool vec = (n & 3) == 0 && (abase & 3) == 0;

    load_slab_rows<GD>(dNs, C::LDZ, dE + static_cast<size_t>(node0) * HD + colbase, HD, n, k8);
    for (int idx = tid; idx < k8 * (TL_ROWS / 4); idx += TL_THREADS) {   // 8 lanes per row of the tile: 128-byte reads
        const int i = idx >> 3, c4 = (idx & 7) * 4;
        float* dst = AsU + i * LDU + c4;
        const float* src = Ab + static_cast<size_t>(i) * n + j0 + c4;
        if (i < n && vec && j0 + c4 < n) {
            tl_cp16(dst, src);
        } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) dst[e] = (i < n && j0 + c4 + e < n) ? src[e] : 0.f;
        }
    }
    tl_cp_wait_all();
    __syncthreads();

    const int mt = warp >> 2, ng = warp & 3;
    float c[C::NT][4];
    zero_frag<C::NT>(c);
    warp_gemm_at<C::NT>(c, k8 / 8, AsU + 16 * mt, LDU, dNs + 8 * C::NT * ng, C::LDZ);
    __syncthreads();                                         // both operand tiles are consumed
    // push-down operands take over the buffer at offsets that do not depend on this document's size:
    // Wt [l GD][LDB] (rows m GD + c' of Wn_l's dense-connect part, B^T operand), then Tt [32][LDB] = dZ_l of the tile
    float* Wt = smem;
    float* Tt = smem + l * GD * C::LDB;
    const float* wsrc = Winner + (static_cast<size_t>(h) * layers + l) * S * GD;
    for (int idx = tid; idx < l * GD * C::CG; idx += TL_THREADS) {
        const int r = idx / C::CG, c4 = (idx - r * C::CG) * 4;
        tl_cp16(Wt + r * C::LDB + c4, wsrc + static_cast<size_t>(r) * GD + c4);
    }
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int jj = 16 * mt + g + 8 * half, j = j0 + jj;
#pragma unroll
        for (int nt = 0; nt < C::NT; ++nt) {
            const int cw = 8 * C::NT * ng + 8 * nt + 2 * t;
            const float2 v = make_float2(c[nt][2 * half], c[nt][2 * half + 1]);
            if (l > 0) *reinterpret_cast<float2*>(Tt + jj * C::LDB + cw) = v;
            if (j < n) *reinterpret_cast<float2*>(dZ + static_cast<size_t>(node0 + j) * HD + colbase + cw) = v;
        }
    }
    if (l == 0) return;
    // dG_m[j][c'] (+)= sum_c dZ_l[j][c] Wn_l[128 + m GD + c'][c]  for m < l  (the slab of dZ that sub-layer m reads);
    // what is accumulated onto is fetched before the product
    float2 cur[2][C::NT];
    tl_cp_wait_all();
    __syncthreads();
    for (int m = 0; m < l; ++m) {
#pragma unroll
        for (int half = 0; half < 2; ++half)
#pragma unroll
            for (int nt = 0; nt < C::NT; ++nt) {
                const int j = j0 + 16 * mt + g + 8 * half;
                cur[half][nt] = make_float2(0.f, 0.f);
                if (l != layers - 1 && j < n)
                    cur[half][nt] = *reinterpret_cast<const float2*>(dZ + static_cast<size_t>(node0 + j) * HD +
                                                                     static_cast<size_t>(h) * S + m * GD +
                                                                     8 * C::NT * ng + 8 * nt + 2 * t);
            }
        zero_frag<C::NT>(c);
        warp_gemm<C::NT, true>(c, GD / 8, Tt + (16 * mt) * C::LDB, C::LDB, Wt + (m * GD + 8 * C::NT * ng) * C::LDB, C::LDB);
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int j = j0 + 16 * mt + g + 8 * half;
            if (j >= n) continue;
#pragma unroll
            for (int nt = 0; nt < C::NT; ++nt) {
                float* p = dZ + static_cast<size_t>(node0 + j) * HD + static_cast<size_t>(h) * S + m * GD +
                           8 * C::NT * ng + 8 * nt + 2 * t;
                *reinterpret_cast<float2*>(p) = make_float2(c[nt][2 * half] + cur[half][nt].x,
                                                            c[nt][2 * half + 1] + cur[half][nt].y);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------
static size_t tile_fwd_smem(int n, int layers, int gd) {
    const int k8 = (n + 7) & ~7, s = layers * gd;
    const size_t tile = static_cast<size_t>(TL_ROWS) * std::max(k8 + 4, s + 4);
    const int kin = (layers - 1) * gd;                                       // recycled: Ws [kin][gd+8] + Gt [32][kin+4]
    const size_t recycled = static_cast<size_t>(kin) * (gd + 8) + static_cast<size_t>(TL_ROWS) * (kin + 4);
    return std::max(static_cast<size_t>(k8) * (gd + 8) + tile + TL_ROWS, recycled) * sizeof(float);
}
static size_t tile_rows_smem(int n, int gd) {
    const int n64 = (n + 63) & ~63;
    return (static_cast<size_t>(n64 + 64) * (gd + 4) + 2 * 64) * sizeof(float);
}
static size_t tile_cols_smem(int n, int layers, int gd) {
    const int k8 = (n + 7) & ~7;
    const size_t recycled = static_cast<size_t>((layers - 1) * gd + TL_ROWS) * (gd + 4);   // Wt + Tt
    return std::max(static_cast<size_t>(k8) * (gd + 8) + static_cast<size_t>(k8) * (TL_ROWS + 8), recycled) * sizeof(float);
}

// graphs of up to 256 entities with sub-layer width 32 or 64 (the document index is blockIdx.z)
bool stack_tiled_usable(const gcgcn_batch* bt, int layers, int slab) {
    if (layers < 1 || slab % layers != 0) return false;
    const int gd = slab / layers;
    return bt->max_nodes <= 256 && bt->num_docs <= 65535 && (gd == 32 || gd == 64);
}

int launch_stack_fwd_tiled(const gcgcn_batch* bt, int heads, int layers, int slab, int flags, const float* A,
                           float* Z, const float* E, const float* Winner, const float* keep, const float* x,
                           float* G, float* F, cudaStream_t st) {
    const int gd = slab / layers, nmax = bt->max_nodes;
    const long long* pp = reinterpret_cast<const long long*>(bt->pair_ptr);
    const dim3 grid(ceil_div(nmax, TL_ROWS), heads, bt->num_docs);
    const size_t smem = tile_fwd_smem(nmax, layers, gd);
    if (gd == 64) GCGCN_TRY(set_smem(stack_tile_fwd_kernel<64>, smem, "stack_tile_fwd"));
    else GCGCN_TRY(set_smem(stack_tile_fwd_kernel<32>, smem, "stack_tile_fwd"));
    for (int l = 0; l < layers; ++l) {
        if (gd == 64)
            stack_tile_fwd_kernel<64><<<grid, TL_THREADS, smem, st>>>(bt->node_ptr, pp, A, Z, E, Winner, keep, x, G, F, l,
                                                                     layers, heads, flags, bt->total_pairs);
        else
            stack_tile_fwd_kernel<32><<<grid, TL_THREADS, smem, st>>>(bt->node_ptr, pp, A, Z, E, Winner, keep, x, G, F, l,
                                                                     layers, heads, flags, bt->total_pairs);
        GCGCN_CHECK_LAUNCH("gcn_stack_tile_fwd");
    }
    return GCGCN_OK;
}

int launch_stack_bwd_tiled(const gcgcn_batch* bt, int heads, int layers, int slab, int flags, const float* A,
                           const float* Z, const float* G, const float* Winner, const float* keep, const float* dF,
                           float* dZ, float* dE, float* dA, cudaStream_t st) {
    const int gd = slab / layers, nmax = bt->max_nodes;
    const long long* pp = reinterpret_cast<const long long*>(bt->pair_ptr);
    const dim3 grid(ceil_div(nmax, TL_ROWS), heads, bt->num_docs);
    const dim3 grid_r(ceil_div(nmax, 64), heads, bt->num_docs);
    const size_t smem_r = tile_rows_smem(nmax, gd), smem_c = tile_cols_smem(nmax, layers, gd);
    if (gd == 64) {
        GCGCN_TRY(set_smem(stack_tile_bwd_rows_kernel<64>, smem_r, "stack_tile_bwd_rows"));
        GCGCN_TRY(set_smem(stack_tile_bwd_cols_kernel<64>, smem_c, "stack_tile_bwd_cols"));
    } else {
        GCGCN_TRY(set_smem(stack_tile_bwd_rows_kernel<32>, smem_r, "stack_tile_bwd_rows"));
        GCGCN_TRY(set_smem(stack_tile_bwd_cols_kernel<32>, smem_c, "stack_tile_bwd_cols"));
    }
    for (int l = layers - 1; l >= 0; --l) {
        if (gd == 64)
            stack_tile_bwd_rows_kernel<64><<<grid_r, TL_THREADS, smem_r, st>>>(bt->node_ptr, pp, A, Z, G, keep, dF, dZ, dE,
                                                                           dA, l, layers, heads, flags, bt->total_pairs);
        else
            stack_tile_bwd_rows_kernel<32><<<grid_r, TL_THREADS, smem_r, st>>>(bt->node_ptr, pp, A, Z, G, keep, dF, dZ, dE,
                                                                           dA, l, layers, heads, flags, bt->total_pairs);
        GCGCN_CHECK_LAUNCH("gcn_stack_tile_bwd_rows");
        if (gd == 64)
            stack_tile_bwd_cols_kernel<64><<<grid, TL_THREADS, smem_c, st>>>(bt->node_ptr, pp, A, Winner, dE, dZ, l, layers,
                                                                           heads, bt->total_pairs);
        else
            stack_tile_bwd_cols_kernel<32><<<grid, TL_THREADS, smem_c, st>>>(bt->node_ptr, pp, A, Winner, dE, dZ, l, layers,
                                                                           heads, bt->total_pairs);
        GCGCN_CHECK_LAUNCH("gcn_stack_tile_bwd_cols");
    }
    return GCGCN_OK;
}

// ---------------------------------------------------------------------------------------------------
// MHA backward for large graphs: dq_h[tile] = scale (dS + dS^T)[tile, :] q_h   (G:136-138 backward; key = query).
// attention.cu's kernel walks dS^T with stride-n scalar reads (32 lines per warp instruction) and gives a whole
// (document, head) to one CTA; here a CTA takes 32 rows, reads its row tile dS[tile, :] and its column tile
// dS[:, tile] as they lie in memory (16-byte async copies) and runs both products on the tensor cores, the second
// one with transposed-A fragment loads.
template <int DH>
__global__ void __launch_bounds__(TL_THREADS, 2)
mha_bwd_tile_kernel(const int* __restrict__ node_ptr, const long long* __restrict__ pair_ptr,
                    const float* __restrict__ q, const float* __restrict__ dS, float* __restrict__ dq,
                    long long total_pairs, float scale) {
    extern __shared__ __align__(16) float smem[];
    const int b = blockIdx.z, h = blockIdx.y, i0 = blockIdx.x * TL_ROWS;
    const int node0 = node_ptr[b];
    const int n = node_ptr[b + 1] - node0;
    if (i0 >= n) return;
    const int k8 = (n + 7) & ~7, lda = k8 + 4;
    constexpr int LDQ = DH + 8, LDU = TL_ROWS + 8;

    float* Qs = smem;                                        // [k8][LDQ]   q_h, all rows
    float* As = Qs + static_cast<size_t>(k8) * LDQ;          // [32][lda]   dS[tile, :]
    float* AsU = As + TL_ROWS * lda;                         // [k8][LDU]   dS[:, tile]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const long long abase = static_cast<long long>(h) * total_pairs + pair_ptr[b];
    const float* Sb = dS + abase;
    const bool vec = (n & 3) == 0 && (abase & 3) == 0;

    for (int idx = tid; idx < k8 * (DH / 4); idx += TL_THREADS) {
        const int j = idx / (DH / 4), c4 = (idx - j * (DH / 4)) * 4;
        if (j < n) tl_cp16(Qs + j * LDQ + c4, q + static_cast<size_t>(node0 + j) * D + h * DH + c4);
        else tl_zero4(Qs + j * LDQ + c4);
    }
    load_att_rows(As, lda, Sb, n, k8, i0, vec);
    for (int idx = tid; idx < k8 * (TL_ROWS / 4); idx += TL_THREADS) {
        const int i = idx >> 3, c4 = (idx & 7) * 4;
        float* dst = AsU + i * LDU + c4;
        const float* src = Sb + static_cast<size_t>(i) * n + i0 + c4;
        if (i < n && vec && i0 + c4 < n) {
            tl_cp16(dst, src);
        } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) dst[e] = (i < n && i0 + c4 + e < n) ? src[e] : 0.f;
        }
    }
    tl_cp_wait_all();
    __syncthreads();

    const int mt = warp & 1, ng = warp >> 1;                 // 2 row tiles x up to 4 column tiles of 8
    if (ng >= DH / 8) return;
    float c[1][4];
    zero_frag<1>(c);
    warp_gemm<1, false>(c, k8 / 8, As + (16 * mt) * lda, lda, Qs + 8 * ng, LDQ);
    warp_gemm_at<1>(c, k8 / 8, AsU + 16 * mt, LDU, Qs + 8 * ng, LDQ);
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int i = i0 + 16 * mt + g + 8 * half;
        if (i >= n) continue;
        *reinterpret_cast<float2*>(dq + static_cast<size_t>(node0 + i) * D + h * DH + 8 * ng + 2 * t) =
            make_float2(c[0][2 * half] * scale, c[0][2 * half + 1] * scale);
    }
}

bool mha_bwd_tiled_usable(const gcgcn_batch* bt, int heads) {
    const int dh = D / heads;
    return bt->max_nodes > 64 && bt->max_nodes <= 256 && bt->num_docs <= 65535 && (dh == 16 || dh == 32);
}

int launch_mha_bwd_tiled(const gcgcn_batch* bt, int heads, const float* q, const float* dS, float* dq,
                         cudaStream_t st) {
    const int dh = D / heads, nmax = bt->max_nodes, k8 = (nmax + 7) & ~7;
    const float scale = 1.0f / sqrtf(static_cast<float>(dh));
    const size_t smem = (static_cast<size_t>(k8) * (dh + 8) + static_cast<size_t>(TL_ROWS) * (k8 + 4) +
                         static_cast<size_t>(k8) * (TL_ROWS + 8)) * sizeof(float);
    const dim3 grid(ceil_div(nmax, TL_ROWS), heads, bt->num_docs);
    const long long* pp = reinterpret_cast<const long long*>(bt->pair_ptr);
    if (dh == 16) {
        GCGCN_TRY(set_smem(mha_bwd_tile_kernel<16>, smem, "mha_bwd_tile"));
        mha_bwd_tile_kernel<16><<<grid, TL_THREADS, smem, st>>>(bt->node_ptr, pp, q, dS, dq, bt->total_pairs, scale);
    } else {
        GCGCN_TRY(set_smem(mha_bwd_tile_kernel<32>, smem, "mha_bwd_tile"));
        mha_bwd_tile_kernel<32><<<grid, TL_THREADS, smem, st>>>(bt->node_ptr, pp, q, dS, dq, bt->total_pairs, scale);
    }
    GCGCN_CHECK_LAUNCH("mha_bwd_tile");
    return GCGCN_OK;
}

}  // namespace gcgcn
