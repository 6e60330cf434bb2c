// Densely connected GraphConv stack (G:36-50 inside G:67-76 / G:103-113), one CTA per
// (document, head).
//
// Per head h and sub-layer l (g = 128 / layers):
//   Z_l  = x Wn_l[0:128] + sum_{m<l} g_m Wn_l[128+m*g : 128+(m+1)*g]      (chain_matmul, G:42)
//   out  = ( ebar We_l + A Z_l ) / r ,  r_i = sum_j A_ij + [sum_j A_ij == 0]   (G:43-50)
//   g_l  = relu(out) ; F = cat_l(keep * g_l) + x                           (G:71-76)
// The two projections over *all* node rows of the batch (x Wn[0:128], ebar We) are dense GEMMs
// done by the caller; they arrive as Zx (in `Z`, updated in place to the final Z_l) and `E`.
// This kernel owns everything that couples the rows of one document: A Z_l, the row
// normalisation, relu, the dense-connect recurrence and the residual.  The n x n map is streamed
// through shared memory in 64-row tiles, so n up to 256 fits one CTA.
//
// The three O(n^2 g) products -- A Z_l forward, dN Z^T and A^T dN backward -- run on the tensor cores
// (mma.sync m16n8k8 TF32 with the 3xTF32 split of mma_tf32.cuh, fp32 parity); the row-local O(n g^2)
// dense-connect products and the element-wise epilogues stay on the CUDA cores.
//
// launch_stack_fwd / launch_stack_bwd choose one of three kernel families from the shape alone:
//   gcn_block.cu        the block configuration (slab 128, ReLU + residual, no keep mask) on graphs of n <= 64;
//   gcn_stack_tiled.cu  otherwise, sub-layer width 32 or 64 with n <= 256 and at most 65,535 documents;
//   this file           everything else: sub-layer width 16 or 128, n > 256, or more than 65,535 documents.
#include "common.cuh"
#include "mma_tf32.cuh"

namespace gcgcn {

constexpr int ST_THREADS = 256;
constexpr int ST_TR = 64;  // attention rows per shared-memory tile

template <int GD>
struct StackCfg {
    static constexpr int CG = GD / 4;            // 4-column groups per sub-layer slab
    static constexpr int NRG = ST_THREADS / CG;  // row groups
    static constexpr int RT = ST_TR / NRG;       // rows per thread
    static constexpr int LDZ = GD + 8;           // forward Z tile: stride == 8 (mod 32), conflict-free B fragments
    static constexpr int LDB = GD + 4;           // backward dN / Z tiles: stride == 4 (mod 8), A and B^T fragments
    static constexpr int NT = GD / 16;           // 8-column MMA tiles per warp (4 row tiles x 2 column groups)
    static_assert(RT >= 1 && RT * NRG == ST_TR, "tile shape");
};

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void fma4(float4& acc, float s, const float4& w) {
    acc.x = fmaf(s, w.x, acc.x); acc.y = fmaf(s, w.y, acc.y);
    acc.z = fmaf(s, w.z, acc.z); acc.w = fmaf(s, w.w, acc.w);
}
__device__ __forceinline__ float dot4(const float4& a, const float4& b) {
    return fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, a.w * b.w)));
}

// load rows [row0, row0+ST_TR) of the document's n x n map into As[ST_TR][lda]; rows >= n are zero
// (columns n .. k8-1, the K padding of the MMA loop, are zero as well)
__device__ __forceinline__ void load_att_tile(float* As, int lda, const float* __restrict__ Ab, int n,
                                              int row0) {
    const int rows = min(ST_TR, n - row0);
    const int k8 = (n + 7) & ~7;
    for (int t = threadIdx.x; t < ST_TR * k8; t += ST_THREADS) {
        int ii = t / k8, j = t - ii * k8;
        As[ii * lda + j] = (ii < rows && j < n) ? Ab[static_cast<size_t>(row0 + ii) * n + j] : 0.f;
    }
}

// the same tile transposed, AsT[j][ii] = A[row0 + ii][j] for j < np16 (zero outside the document)
__device__ __forceinline__ void load_att_tile_t(float* AsT, int ldt, const float* __restrict__ Ab, int n,
                                                int row0, int np16) {
    const int rows = min(ST_TR, n - row0);
    for (int t = threadIdx.x; t < ST_TR * np16; t += ST_THREADS) {
        int ii = t / np16, j = t - ii * np16;
        AsT[j * ldt + ii] = (ii < rows && j < n) ? Ab[static_cast<size_t>(row0 + ii) * n + j] : 0.f;
    }
}

// r_i = rowsum(A) + [rowsum == 0]     (G:47-49), one warp per row straight from global memory
__device__ __forceinline__ void row_norms(float* rs, const float* __restrict__ Ab, int n) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = warp; i < n; i += ST_THREADS / WARP) {
        float s = 0.f;
        for (int j = lane; j < n; j += WARP) s += Ab[static_cast<size_t>(i) * n + j];
        s = warp_sum(s);
        if (lane == 0) rs[i] = s + (s == 0.f ? 1.f : 0.f);
    }
}

// ---------------------------------------------------------------------------------------------
template <int GD>
__global__ void __launch_bounds__(ST_THREADS)
gcn_stack_fwd_kernel(const int* __restrict__ node_ptr, const long long* __restrict__ pair_ptr,
                     const float* __restrict__ A, float* __restrict__ Z, const float* __restrict__ E,
                     const float* __restrict__ Winner, const float* __restrict__ keep,
                     const float* __restrict__ x, float* __restrict__ G, float* __restrict__ F,
                     int layers, int heads, int flags, long long total_pairs) {
    using C = StackCfg<GD>;
    extern __shared__ __align__(16) float smem[];
    const int b = blockIdx.x, h = blockIdx.y;
    const int node0 = node_ptr[b];
    const int n = node_ptr[b + 1] - node0;
    if (n == 0) return;
    const int S = layers * GD;   // per-head slab width (= 128 inside the conv blocks)
    const int HD = heads * S;
    const int KI = (layers - 1) * GD;
    const int LDG = KI + 1;
    const int k8 = (n + 7) & ~7;        // K of the A Z_l product, zero padded
    const int lda = k8 + 4;             // == 4 (mod 8): conflict-free A fragments
    const int ntiles = (n + ST_TR - 1) / ST_TR;
    const int npad = ntiles * ST_TR;

    float* Zl = smem;                                      // [npad][LDZ]
    float* Gs = Zl + static_cast<size_t>(npad) * C::LDZ;   // [n][LDG]
    float* As = Gs + static_cast<size_t>(n) * LDG;         // [ST_TR][lda]
    float* Wl = As + static_cast<size_t>(ST_TR) * lda;     // [KI][GD]
    Wl = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(Wl) + 15) & ~uintptr_t(15));
    float* rs = Wl + static_cast<size_t>(KI) * GD;         // [n]

    const float* Ab = A + static_cast<long long>(h) * total_pairs + pair_ptr[b];
    const int cg = threadIdx.x % C::CG, rg = threadIdx.x / C::CG;
    const int c0 = cg * 4;
    const bool relu = flags & GCGCN_STACK_RELU, resid = flags & GCGCN_STACK_RESIDUAL;

    row_norms(rs, Ab, n);

    for (int l = 0; l < layers; ++l) {
        const int kin = l * GD;  // dense-connect inputs available to this sub-layer
        if (l > 0) {
            const float* wsrc = Winner + (static_cast<size_t>(h) * layers + l) * S * GD;
            for (int t = threadIdx.x * 4; t < kin * GD; t += ST_THREADS * 4) st4(Wl + t, ld4(wsrc + t));
        }
        __syncthreads();
        // (1) Z_l rows = Zx rows + g_{<l} rows x Winner  (row-local)
        const size_t col = static_cast<size_t>(h) * S + l * GD + c0;
        for (int pb = 0; pb < ntiles; ++pb) {
            float4 acc[C::RT];
            int rows[C::RT];
#pragma unroll
            for (int a = 0; a < C::RT; ++a) {
                rows[a] = pb * ST_TR + rg * C::RT + a;
                acc[a] = rows[a] < n ? ld4(Z + static_cast<size_t>(node0 + rows[a]) * HD + col)
                                     : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            for (int k = 0; k < kin; ++k) {
                float4 w = ld4(Wl + k * GD + c0);
#pragma unroll
                for (int a = 0; a < C::RT; ++a) {
                    float gk = Gs[min(rows[a], n - 1) * LDG + k];
                    fma4(acc[a], gk, w);
                }
            }
#pragma unroll
            for (int a = 0; a < C::RT; ++a) {
                if (rows[a] >= n) acc[a] = make_float4(0.f, 0.f, 0.f, 0.f);  // padding rows stay zero
                st4(Zl + rows[a] * C::LDZ + c0, acc[a]);
                if (rows[a] < n && l > 0) st4(Z + static_cast<size_t>(node0 + rows[a]) * HD + col, acc[a]);
            }
        }
        __syncthreads();
        // (2) out rows = (E + A Z_l) / r, tile of 64 attention rows at a time on the tensor cores:
        //     warp (mt, ng) owns rows 16 mt .. 16 mt + 15 of the tile and columns ng * GD/2 .. + GD/2 - 1
        {
            const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
            const int mt = warp >> 1, ng = warp & 1;
            const size_t colbase = static_cast<size_t>(h) * S + l * GD;
            for (int pb = 0; pb < ntiles; ++pb) {
                load_att_tile(As, lda, Ab, n, pb * ST_TR);
                __syncthreads();
                float c[C::NT][4];
                zero_frag<C::NT>(c);
                warp_gemm<C::NT, false>(c, k8 / 8, As + (16 * mt) * lda, lda, Zl + 8 * C::NT * ng, C::LDZ);
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    const int i = pb * ST_TR + 16 * mt + g + 8 * half;
                    if (i >= n) continue;
                    const float r = rs[i];
#pragma unroll
                    for (int nt = 0; nt < C::NT; ++nt) {
                        const int cw = 8 * C::NT * ng + 8 * nt + 2 * t;
                        const size_t off = static_cast<size_t>(node0 + i) * HD + colbase + cw;
                        const float2 e2 = ld2g(E + off);
                        float2 o;
                        o.x = (e2.x + c[nt][2 * half]) / r;
                        o.y = (e2.y + c[nt][2 * half + 1]) / r;
                        if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); }
                        *reinterpret_cast<float2*>(G + off) = o;
                        if (l < layers - 1) {
                            float* gs = Gs + i * LDG + kin + cw;
                            gs[0] = o.x; gs[1] = o.y;
                        }
                        float2 f = o;
                        if (keep != nullptr) { const float2 k2 = ld2g(keep + off); f.x *= k2.x; f.y *= k2.y; }
                        if (resid) {
                            const float2 x2 = ld2g(x + static_cast<size_t>(node0 + i) * S + l * GD + cw);
                            f.x += x2.x; f.y += x2.y;
                        }
                        *reinterpret_cast<float2*>(F + off) = f;
                    }
                }
                __syncthreads();
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// backward of the stack.  Inputs: dF (grad of F; the residual's share of dx is added by the
// caller), saved Z, G, A.  Outputs: dZ (grad of Zx -- equals grad of Z_l), dE, dA.
// Sub-layers are walked top-down.  Gradients that later sub-layers send to g_m through the dense
// connection are accumulated in dZ's own column slab m, which is free until sub-layer m is
// processed (then it is consumed and overwritten with dZ_m).
template <int GD>
__global__ void __launch_bounds__(ST_THREADS)
gcn_stack_bwd_kernel(const int* __restrict__ node_ptr, const long long* __restrict__ pair_ptr,
                     const float* __restrict__ A, const float* __restrict__ Z,
                     const float* __restrict__ G, const float* __restrict__ Winner,
                     const float* __restrict__ keep, const float* __restrict__ dF,
                     float* __restrict__ dZ, float* __restrict__ dE, float* __restrict__ dA,
                     int layers, int heads, int flags, long long total_pairs) {
    using C = StackCfg<GD>;
    extern __shared__ __align__(16) float smem[];
    const int b = blockIdx.x, h = blockIdx.y;
    const int node0 = node_ptr[b];
    const int n = node_ptr[b + 1] - node0;
    if (n == 0) return;
    const int S = layers * GD;   // per-head slab width (= 128 inside the conv blocks)
    const int HD = heads * S;
    const int np16 = (n + 15) & ~15;    // M of the A^T dN product
    constexpr int LDT = ST_TR + 4;      // transposed attention tile: == 4 (mod 8)
    const int ntiles = (n + ST_TR - 1) / ST_TR;
    const int npad = ntiles * ST_TR;

    float* dNs = smem;                                       // [npad][LDZ]  dN_l = dOut / r
    float* Ts = dNs + static_cast<size_t>(npad) * C::LDB;    // [npad][LDZ]  Z_l, later dZ_l
    float* WT = Ts + static_cast<size_t>(npad) * C::LDB;     // [(layers-1)][GD][GD] transposed slices
    float* AsT = WT + static_cast<size_t>(layers - 1) * GD * GD;  // [np16][LDT]  AsT[j][ii] = A[tile row ii][j]
    float* rs = AsT + static_cast<size_t>(np16) * LDT;       // [n]
    float* drs = rs + n;                                     // [n]

    const long long abase = static_cast<long long>(h) * total_pairs + pair_ptr[b];
    const float* Ab = A + abase;
    float* dAb = dA + abase;
    const int cg = threadIdx.x % C::CG, rg = threadIdx.x / C::CG;
    const int c0 = cg * 4;
    const bool relu = flags & GCGCN_STACK_RELU;

    row_norms(rs, Ab, n);
    for (int t = threadIdx.x; t < n; t += ST_THREADS) drs[t] = 0.f;
    __syncthreads();

    for (int l = layers - 1; l >= 0; --l) {
        const size_t col = static_cast<size_t>(h) * S + l * GD + c0;
        // WT[m][c][c'] = Wn_l[128 + m*GD + c'][c]  for m < l  (transposed for conflict-free reads)
        if (l > 0) {
            const float* wsrc = Winner + (static_cast<size_t>(h) * layers + l) * S * GD;
            for (int t = threadIdx.x; t < l * GD * GD; t += ST_THREADS) {
                int m = t / (GD * GD), rem = t - m * GD * GD;
                int cp = rem / GD, c = rem - cp * GD;  // wsrc[(m*GD + cp)*GD + c]
                WT[(m * GD + c) * GD + cp] = wsrc[t];
            }
        }
        // (a) row-local: dG_l -> dOut -> dN_l, dE_l, dr
        for (int pb = 0; pb < ntiles; ++pb) {
#pragma unroll
            for (int a = 0; a < C::RT; ++a) {
                const int i = pb * ST_TR + rg * C::RT + a;
                float4 dn = make_float4(0.f, 0.f, 0.f, 0.f);
                float4 zl = make_float4(0.f, 0.f, 0.f, 0.f);
                float drp = 0.f;
                if (i < n) {
                    const size_t off = static_cast<size_t>(node0 + i) * HD + col;
                    float4 dg = ld4(dF + off);
                    if (keep != nullptr) {
                        const float4 k4 = ld4(keep + off);
                        dg.x *= k4.x; dg.y *= k4.y; dg.z *= k4.z; dg.w *= k4.w;
                    }
                    if (l < layers - 1) {
                        const float4 s4 = ld4(dZ + off);
                        dg.x += s4.x; dg.y += s4.y; dg.z += s4.z; dg.w += s4.w;
                    }
                    const float4 g4 = ld4(G + off);
                    if (relu) {
                        dg.x = g4.x > 0.f ? dg.x : 0.f; dg.y = g4.y > 0.f ? dg.y : 0.f;
                        dg.z = g4.z > 0.f ? dg.z : 0.f; dg.w = g4.w > 0.f ? dg.w : 0.f;
                    }
                    const float r = rs[i];
                    dn.x = dg.x / r; dn.y = dg.y / r; dn.z = dg.z / r; dn.w = dg.w / r;
                    st4(dE + off, dn);
                    drp = -(dn.x * g4.x + dn.y * g4.y + dn.z * g4.z + dn.w * g4.w);
                    zl = ld4(Z + off);
                }
                st4(dNs + (pb * ST_TR + rg * C::RT + a) * C::LDB + c0, dn);
                st4(Ts + (pb * ST_TR + rg * C::RT + a) * C::LDB + c0, zl);
#pragma unroll
                for (int o = C::CG / 2; o > 0; o >>= 1) drp += __shfl_xor_sync(0xffffffffu, drp, o);
                if (cg == 0 && i < n) drs[i] += drp;
            }
        }
        __syncthreads();
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
        // (c) dA rows += dN_l Z_l^T (+ dr at the last processed sub-layer): 64 x 64 blocks on the tensor cores,
        //     warp (mt, ng) owns rows 16 mt .. + 15 and columns 32 ng .. + 31 of a block
        {
            const int mt = warp >> 1, ng = warp & 1;
            for (int pb = 0; pb < ntiles; ++pb) {
                for (int jp = 0; jp < ntiles; ++jp) {
                    float c[4][4];
                    zero_frag<4>(c);
                    warp_gemm<4, true>(c, GD / 8, dNs + (pb * ST_TR + 16 * mt) * C::LDB, C::LDB,
                                       Ts + (jp * ST_TR + 32 * ng) * C::LDB, C::LDB);
#pragma unroll
                    for (int half = 0; half < 2; ++half) {
                        const int i = pb * ST_TR + 16 * mt + g + 8 * half;
                        if (i >= n) continue;
                        const float dr = (l == 0) ? drs[i] : 0.f;
#pragma unroll
                        for (int nt = 0; nt < 4; ++nt) {
#pragma unroll
                            for (int e = 0; e < 2; ++e) {
                                const int j = jp * ST_TR + 32 * ng + 8 * nt + 2 * t + e;
                                if (j >= n) continue;
                                float* p = dAb + static_cast<size_t>(i) * n + j;
                                float val = c[nt][2 * half + e] + dr;
                                if (l != layers - 1) val += *p;
                                *p = val;
                            }
                        }
                    }
                }
            }
        }
        __syncthreads();
        // (b) dZ_l = A^T dN_l, accumulated over attention tiles into Ts (Z_l is no longer needed): per tile,
        //     C[j][c] += sum_ii AsT[j][ii] dN[tile row ii][c]; unit u = (row tile of j, column group) stays with
        //     one warp over all tiles, so the read-modify-write of Ts needs no extra barrier
        for (int idx = threadIdx.x; idx < npad * C::LDB; idx += ST_THREADS) Ts[idx] = 0.f;
        for (int pb = 0; pb < ntiles; ++pb) {
            __syncthreads();
            load_att_tile_t(AsT, LDT, Ab, n, pb * ST_TR, np16);
            __syncthreads();
            for (int u = warp; u < (np16 / 16) * 2; u += ST_THREADS / WARP) {
                const int mt = u >> 1, ng = u & 1;
                float* tc = Ts + (16 * mt) * C::LDB + 8 * C::NT * ng;
                float c[C::NT][4];
#pragma unroll
                for (int nt = 0; nt < C::NT; ++nt) {
                    const float2 lo = *reinterpret_cast<const float2*>(tc + g * C::LDB + 8 * nt + 2 * t);
                    const float2 hi = *reinterpret_cast<const float2*>(tc + (g + 8) * C::LDB + 8 * nt + 2 * t);
                    c[nt][0] = lo.x; c[nt][1] = lo.y; c[nt][2] = hi.x; c[nt][3] = hi.y;
                }
                warp_gemm<C::NT, false>(c, ST_TR / 8, AsT + (16 * mt) * LDT, LDT,
                                        dNs + (pb * ST_TR) * C::LDB + 8 * C::NT * ng, C::LDB);
#pragma unroll
                for (int nt = 0; nt < C::NT; ++nt) {
                    *reinterpret_cast<float2*>(tc + g * C::LDB + 8 * nt + 2 * t) = make_float2(c[nt][0], c[nt][1]);
                    *reinterpret_cast<float2*>(tc + (g + 8) * C::LDB + 8 * nt + 2 * t) = make_float2(c[nt][2], c[nt][3]);
                }
            }
        }
        __syncthreads();
        // write dZ_l and push its dense-connect share down to the slabs m < l:
        //   dG_m[j][c'] += sum_c dZ_l[j][c] * Wn_l[128 + m*GD + c'][c]
        for (int jp = 0; jp < ntiles; ++jp) {
#pragma unroll
            for (int a = 0; a < C::RT; ++a) {
                const int j = jp * ST_TR + rg * C::RT + a;
                if (j < n)
                    st4(dZ + static_cast<size_t>(node0 + j) * HD + col, ld4(Ts + j * C::LDB + c0));
            }
            for (int m = 0; m < l; ++m) {
                float4 acc[C::RT];
#pragma unroll
                for (int a = 0; a < C::RT; ++a) acc[a] = make_float4(0.f, 0.f, 0.f, 0.f);
                const float* wt = WT + static_cast<size_t>(m) * GD * GD + c0;
                const float* trow = Ts + (jp * ST_TR + rg * C::RT) * C::LDB;
                for (int c = 0; c < GD; ++c) {
                    const float4 w = ld4(wt + c * GD);
#pragma unroll
                    for (int a = 0; a < C::RT; ++a) fma4(acc[a], trow[a * C::LDB + c], w);
                }
#pragma unroll
                for (int a = 0; a < C::RT; ++a) {
                    const int j = jp * ST_TR + rg * C::RT + a;
                    if (j >= n) continue;
                    float* p = dZ + static_cast<size_t>(node0 + j) * HD + static_cast<size_t>(h) * S +
                               m * GD + c0;
                    float4 val = acc[a];
                    if (l != layers - 1) {
                        const float4 cur = ld4(p);
                        val.x += cur.x; val.y += cur.y; val.z += cur.z; val.w += cur.w;
                    }
                    st4(p, val);
                }
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
static size_t stack_fwd_smem(int n, int layers, int gd) {
    int npad = ((n + ST_TR - 1) / ST_TR) * ST_TR;
    int ki = (layers - 1) * gd;
    size_t fl = static_cast<size_t>(npad) * (gd + 8) + static_cast<size_t>(n) * (ki + 1) +
                static_cast<size_t>(ST_TR) * (((n + 7) & ~7) + 4) + 4 + static_cast<size_t>(ki) * gd + n;
    return fl * sizeof(float);
}
static size_t stack_bwd_smem(int n, int layers, int gd) {
    int npad = ((n + ST_TR - 1) / ST_TR) * ST_TR;
    size_t fl = 2 * static_cast<size_t>(npad) * (gd + 4) + static_cast<size_t>(layers - 1) * gd * gd +
                static_cast<size_t>((n + 15) & ~15) * (ST_TR + 4) + 2 * static_cast<size_t>(n);
    return fl * sizeof(float);
}

// row-tiled tensor-core versions for max n <= 256 and sub-layer width 32 or 64, gcn_stack_tiled.cu
bool stack_tiled_usable(const gcgcn_batch* bt, int layers, int slab);
int launch_stack_fwd_tiled(const gcgcn_batch* bt, int heads, int layers, int slab, int flags, const float* A,
                           float* Z, const float* E, const float* Winner, const float* keep, const float* x,
                           float* G, float* F, cudaStream_t st);
int launch_stack_bwd_tiled(const gcgcn_batch* bt, int heads, int layers, int slab, int flags, const float* A,
                           const float* Z, const float* G, const float* Winner, const float* keep, const float* dF,
                           float* dZ, float* dE, float* dA, cudaStream_t st);

bool block_kernels_usable(const gcgcn_batch* bt, int heads, int layers, int slab, bool mha);
int launch_block_fwd(const gcgcn_batch* bt, int heads, int layers, const float* A, const float* q, float* P,
                     float* Z, const float* E, const float* Winner, const float* x, float* G, float* F,
                     float* frag_ws, const BlockDrop& drop, cudaStream_t st);
int launch_block_bwd(const gcgcn_batch* bt, int heads, int layers, int out_mode, const float* A, const float* q,
                     const float* Z, const float* G, const float* Winner, const float* dF, float* dZ, float* dE,
                     float* dOut, float* frag_ws, const BlockDrop& drop, cudaStream_t st);

// the block configuration (ReLU + residual, no dropout mask, slab 128, n <= 64) has its own kernels (gcn_block.cu)
static bool block_config(const gcgcn_batch* bt, int heads, int layers, int slab, int flags, const float* keep) {
    const int need = GCGCN_STACK_RELU | GCGCN_STACK_RESIDUAL;
    return keep == nullptr && (flags & need) == need && block_kernels_usable(bt, heads, layers, slab, false);
}

int launch_stack_fwd(const gcgcn_batch* bt, int heads, int layers, int slab, int flags, const float* A, float* Z,
                     const float* E, const float* Winner, const float* keep, const float* x, float* G,
                     float* F, float* frag_ws, cudaStream_t st) {
    if (bt->num_docs == 0) return GCGCN_OK;
    if (block_config(bt, heads, layers, slab, flags, keep) && (frag_ws != nullptr || layers < 2))
        return launch_block_fwd(bt, heads, layers, A, nullptr, nullptr, Z, E, Winner, x, G, F, frag_ws, BlockDrop{}, st);
    if (stack_tiled_usable(bt, layers, slab))
        return launch_stack_fwd_tiled(bt, heads, layers, slab, flags, A, Z, E, Winner, keep, x, G, F, st);
    if (layers < 1 || slab % layers != 0)
        return fail(GCGCN_ERR_UNSUPPORTED, "layer_num %d must divide the output width %d", layers, slab);
    const int gd = slab / layers;
    const size_t smem = stack_fwd_smem(bt->max_nodes, layers, gd);
    dim3 grid(bt->num_docs, heads);
    const long long* pp = reinterpret_cast<const long long*>(bt->pair_ptr);
#define GCGCN_STACK_FWD(GDV)                                                                        \
    case GDV:                                                                                       \
        GCGCN_TRY(set_smem(gcn_stack_fwd_kernel<GDV>, smem, "gcn_stack_fwd"));                      \
        gcn_stack_fwd_kernel<GDV><<<grid, ST_THREADS, smem, st>>>(bt->node_ptr, pp, A, Z, E, Winner, \
                                                                   keep, x, G, F, layers, heads,    \
                                                                   flags, bt->total_pairs);         \
        break;
    switch (gd) {
        GCGCN_STACK_FWD(16)
        GCGCN_STACK_FWD(32)
        GCGCN_STACK_FWD(64)
        GCGCN_STACK_FWD(128)
        default:
            return fail(GCGCN_ERR_UNSUPPORTED, "sub-layer width g = %d (layer_num %d) not supported; g must be 16, 32, 64 or 128",
                        gd, layers);
    }
#undef GCGCN_STACK_FWD
    GCGCN_CHECK_LAUNCH("gcn_stack_fwd");
    return GCGCN_OK;
}

int launch_stack_bwd(const gcgcn_batch* bt, int heads, int layers, int slab, int flags, const float* A,
                     const float* Z, const float* G, const float* Winner, const float* keep,
                     const float* dF, float* dZ, float* dE, float* dA, float* frag_ws, cudaStream_t st) {
    if (bt->num_docs == 0) return GCGCN_OK;
    if (block_config(bt, heads, layers, slab, flags, keep) && (frag_ws != nullptr || layers < 2))
        return launch_block_bwd(bt, heads, layers, /*BK_OUT_DA*/ 0, A, nullptr, Z, G, Winner, dF, dZ, dE, dA, frag_ws,
                                BlockDrop{}, st);
    if (stack_tiled_usable(bt, layers, slab))
        return launch_stack_bwd_tiled(bt, heads, layers, slab, flags, A, Z, G, Winner, keep, dF, dZ, dE, dA, st);
    if (layers < 1 || slab % layers != 0)
        return fail(GCGCN_ERR_UNSUPPORTED, "layer_num %d must divide the output width %d", layers, slab);
    const int gd = slab / layers;
    const size_t smem = stack_bwd_smem(bt->max_nodes, layers, gd);
    dim3 grid(bt->num_docs, heads);
    const long long* pp = reinterpret_cast<const long long*>(bt->pair_ptr);
#define GCGCN_STACK_BWD(GDV)                                                                        \
    case GDV:                                                                                       \
        GCGCN_TRY(set_smem(gcn_stack_bwd_kernel<GDV>, smem, "gcn_stack_bwd"));                      \
        gcn_stack_bwd_kernel<GDV><<<grid, ST_THREADS, smem, st>>>(bt->node_ptr, pp, A, Z, G, Winner, \
                                                                   keep, dF, dZ, dE, dA, layers,    \
                                                                   heads, flags, bt->total_pairs);  \
        break;
    switch (gd) {
        GCGCN_STACK_BWD(16)
        GCGCN_STACK_BWD(32)
        GCGCN_STACK_BWD(64)
        GCGCN_STACK_BWD(128)
        default:
            return fail(GCGCN_ERR_UNSUPPORTED, "sub-layer width g = %d (layer_num %d) not supported; g must be 16, 32, 64 or 128",
                        gd, layers);
    }
#undef GCGCN_STACK_BWD
    GCGCN_CHECK_LAUNCH("gcn_stack_bwd");
    return GCGCN_OK;
}

}  // namespace gcgcn
