// Dense-connected GraphConv stack for DocRED-sized graphs (n <= 64), warp-level tensor-core version.
//
// Same contract as gcn_stack.cu (one CTA per (document, head); see that file for the math), but every
// small per-document product -- A Z_l, g_{<l} Winner, and in backward dN Z^T, A^T dN, dZ Winner^T --
// runs on the tensor cores with mma.sync.m16n8k8 TF32.  fp32 parity (<= 1e-4 abs vs the reference) is
// kept by the same 3xTF32 operand split as the tcgen05 projection GEMM: x = hi + lo with hi exactly
// representable in TF32, and  a*b ~= lo_a*hi_b + hi_a*lo_b + hi_a*hi_b.
//
// Why mma.sync and not tcgen05 here: the matrices belong to ONE document (16..64 rows); a tcgen05 tile
// is 128 rows and would have to be built from several documents' block-diagonal attention maps.  The
// document-batched projections (where M is every node row of the batch) are the tcgen05 kernel's job.
//
// Operands live in shared memory as fp32 and are split in registers after the fragment loads.  Row
// strides are chosen so that both fragment access patterns (lanes = 8 rows x 4 k, or 4 k x 8 cols) are
// bank-conflict free or at worst 2-way.
#include "common.cuh"
#include "mma_tf32.cuh"

namespace gcgcn {

constexpr int SM_THREADS = 128;
constexpr int SM_WARPS = SM_THREADS / WARP;

// ---------------------------------------------------------------------------------------------
template <int GD>
__global__ void __launch_bounds__(SM_THREADS)
stack_fwd_mma_kernel(const int* __restrict__ node_ptr, const long long* __restrict__ pair_ptr,
                     const float* __restrict__ A, float* __restrict__ Z, const float* __restrict__ E,
                     const float* __restrict__ Winner, const float* __restrict__ keep,
                     const float* __restrict__ x, float* __restrict__ G, float* __restrict__ F, int layers,
                     int heads, int flags, long long total_pairs, const int* __restrict__ doc_order, int first) {
    extern __shared__ __align__(16) float smem[];
    const int b = doc_order != nullptr ? doc_order[first + blockIdx.x] : blockIdx.x;
    const int h = blockIdx.y;
    const int node0 = node_ptr[b];
    const int n = node_ptr[b + 1] - node0;
    if (n == 0) return;
    const int S = layers * GD, HD = heads * S, KI = (layers - 1) * GD;
    const int NP = (n + 15) & ~15;
    const int LDA = NP + 4, LDG = KI + 4;
    constexpr int LDZ = GD + 8, NG = GD / 32;

    float* As = smem;                 // [NP][LDA]  attention map, zero padded
    float* Zs = As + NP * LDA;        // [NP][LDZ]  Z_l
    float* Gs = Zs + NP * LDZ;        // [NP][LDG]  g_0 .. g_{L-2}
    float* rs = Gs + NP * LDG;        // [NP]  reciprocal row normalisers
    // The dense-connect weights (16 KB per head) are read as MMA fragments straight from global memory:
    // co-resident CTAs work on the same head, so they stay L1-resident, and leaving them out of shared
    // memory raises occupancy (the kernel is latency-, not bandwidth-bound).

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const float* Ab = A + static_cast<long long>(h) * total_pairs + pair_ptr[b];
    const bool relu = flags & GCGCN_STACK_RELU, resid = flags & GCGCN_STACK_RESIDUAL;

    // attention map -> shared (zero padded), one warp per row, and 1 / (rowsum + [rowsum == 0])   (G:47-49)
    for (int i = warp; i < NP; i += SM_WARPS) {
        float s = 0.f;
        for (int j = lane; j < NP; j += WARP) {
            const float v = (i < n && j < n) ? Ab[static_cast<size_t>(i) * n + j] : 0.f;
            As[i * LDA + j] = v;
            s += v;
        }
        s = warp_sum(s);
        if (lane == 0) rs[i] = 1.0f / (s + (s == 0.f ? 1.f : 0.f));
    }
    for (int idx = tid; idx < NP * LDG; idx += SM_THREADS) Gs[idx] = 0.f;

    const int MT = NP / 16;
    for (int l = 0; l < layers; ++l) {
        const int kin = l * GD;
        const size_t colbase = static_cast<size_t>(h) * S + l * GD;
        const float* wsrc = Winner + (static_cast<size_t>(h) * layers + l) * S * GD;
        for (int idx = tid; idx < NP * (GD / 4); idx += SM_THREADS) {
            const int i = idx / (GD / 4), c4 = (idx - i * (GD / 4)) * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < n) v = ld4g(Z + static_cast<size_t>(node0 + i) * HD + colbase + c4);
            *reinterpret_cast<float4*>(Zs + i * LDZ + c4) = v;
        }
        __syncthreads();
        if (l > 0) {
            // Z_l += g_{<l} Winner_l   (dense connection, row-local in the reference: G:72-73)
            for (int u = warp; u < MT * NG; u += SM_WARPS) {
                const int mt = u / NG, ng = u - mt * NG;
                float c[4][4];
                float* zc = Zs + (16 * mt) * LDZ + 32 * ng;
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) {
                    const float2 lo = *reinterpret_cast<const float2*>(zc + g * LDZ + 8 * nt + 2 * t);
                    const float2 hi = *reinterpret_cast<const float2*>(zc + (g + 8) * LDZ + 8 * nt + 2 * t);
                    c[nt][0] = lo.x; c[nt][1] = lo.y; c[nt][2] = hi.x; c[nt][3] = hi.y;
                }
                const float* ga = Gs + (16 * mt) * LDG;
                const float* wb = wsrc + 32 * ng;
                warp_gemm<4, false>(c, kin / 8, ga, LDG, wb, GD);
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) {
                    *reinterpret_cast<float2*>(zc + g * LDZ + 8 * nt + 2 * t) = make_float2(c[nt][0], c[nt][1]);
                    *reinterpret_cast<float2*>(zc + (g + 8) * LDZ + 8 * nt + 2 * t) = make_float2(c[nt][2], c[nt][3]);
                }
            }
            __syncthreads();
            for (int idx = tid; idx < n * (GD / 4); idx += SM_THREADS) {   // final Z_l, saved for backward
                const int i = idx / (GD / 4), c4 = (idx - i * (GD / 4)) * 4;
                *reinterpret_cast<float4*>(Z + static_cast<size_t>(node0 + i) * HD + colbase + c4) =
                    *reinterpret_cast<const float4*>(Zs + i * LDZ + c4);
            }
        }
        // out = (E + A Z_l) / r ; g_l = relu(out) ; F = keep * g_l + x
        for (int u = warp; u < MT * NG; u += SM_WARPS) {
            const int mt = u / NG, ng = u - mt * NG;
            float c[4][4];
            zero_frag<4>(c);
            const float* aa = As + (16 * mt) * LDA;
            const float* zb = Zs + 32 * ng;
            warp_gemm<4, false>(c, NP / 8, aa, LDA, zb, LDZ);
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int i = 16 * mt + g + 8 * half;
                if (i >= n) continue;
                const float rinv = rs[i];
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) {
                    const int col = 32 * ng + 8 * nt + 2 * t;
                    const size_t off = static_cast<size_t>(node0 + i) * HD + colbase + col;
                    const float2 e2 = ld2g(E + off);
                    float2 o;
                    o.x = (e2.x + c[nt][2 * half]) * rinv;
                    o.y = (e2.y + c[nt][2 * half + 1]) * rinv;
                    if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); }
                    *reinterpret_cast<float2*>(G + off) = o;
                    if (l < layers - 1) *reinterpret_cast<float2*>(Gs + i * LDG + kin + col) = o;
                    float2 f = o;
                    if (keep != nullptr) { const float2 k2 = ld2g(keep + off); f.x *= k2.x; f.y *= k2.y; }
                    if (resid) {
                        const float2 x2 = ld2g(x + static_cast<size_t>(node0 + i) * S + l * GD + col);
                        f.x += x2.x; f.y += x2.y;
                    }
                    *reinterpret_cast<float2*>(F + off) = f;
                }
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
template <int GD>
__global__ void __launch_bounds__(SM_THREADS)
stack_bwd_mma_kernel(const int* __restrict__ node_ptr, const long long* __restrict__ pair_ptr,
                     const float* __restrict__ A, const float* __restrict__ Z, const float* __restrict__ G,
                     const float* __restrict__ Winner, const float* __restrict__ keep,
                     const float* __restrict__ dF, float* __restrict__ dZ, float* __restrict__ dE,
                     float* __restrict__ dA, int layers, int heads, int flags, long long total_pairs,
                     const int* __restrict__ doc_order, int first) {
    extern __shared__ __align__(16) float smem[];
    const int b = doc_order != nullptr ? doc_order[first + blockIdx.x] : blockIdx.x;
    const int h = blockIdx.y;
    const int node0 = node_ptr[b];
    const int n = node_ptr[b + 1] - node0;
    if (n == 0) return;
    const int S = layers * GD, HD = heads * S;
    const int NP = (n + 15) & ~15;
    const int LDA = NP + 4;
    constexpr int LDN = GD + 12, NG = GD / 32, CG = GD / 4, RPP = SM_THREADS / CG;

    float* Ats = smem;                 // [NP][LDA]  A transposed: Ats[j][i] = A[i][j]
    float* dNs = Ats + NP * LDA;       // [NP][LDN]  dN_l = dOut_l / r
    float* Ts = dNs + NP * LDN;        // [NP][LDN]  Z_l, later dZ_l
    float* rs = Ts + NP * LDN;         // [NP]   (dense-connect weights: fragments from global, see fwd)
    float* drs = rs + NP;              // [NP]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const long long abase = static_cast<long long>(h) * total_pairs + pair_ptr[b];
    const float* Ab = A + abase;
    float* dAb = dA + abase;
    const bool relu = flags & GCGCN_STACK_RELU;

    // attention map -> shared, transposed and zero padded; reciprocal row normalisers (G:47-49)
    for (int i = warp; i < NP; i += SM_WARPS) {
        float s = 0.f;
        for (int j = lane; j < NP; j += WARP) {
            const float v = (i < n && j < n) ? Ab[static_cast<size_t>(i) * n + j] : 0.f;
            Ats[j * LDA + i] = v;
            s += v;
        }
        s = warp_sum(s);
        if (lane == 0) { rs[i] = 1.0f / (s + (s == 0.f ? 1.f : 0.f)); drs[i] = 0.f; }
    }
    __syncthreads();

    const int MT = NP / 16;
    const int cg = tid % CG, rg = tid / CG, c0 = cg * 4;
    for (int l = layers - 1; l >= 0; --l) {
        const size_t colbase = static_cast<size_t>(h) * S + l * GD;
        const float* wsrc = Winner + (static_cast<size_t>(h) * layers + l) * S * GD;
        // (a) row-local: dG_l -> dOut -> dN_l (shared), dE_l (global), dr (shared)
        for (int i = rg; i < NP; i += RPP) {
            float4 dn = make_float4(0.f, 0.f, 0.f, 0.f), zl = dn;
            float drp = 0.f;
            if (i < n) {
                const size_t off = static_cast<size_t>(node0 + i) * HD + colbase + c0;
                float4 dg = ld4g(dF + off);
                if (keep != nullptr) {
                    const float4 k4 = ld4g(keep + off);
                    dg.x *= k4.x; dg.y *= k4.y; dg.z *= k4.z; dg.w *= k4.w;
                }
                if (l < layers - 1) {
                    const float4 s4 = ld4g(dZ + off);      // dense-connect gradient parked in slab l
                    dg.x += s4.x; dg.y += s4.y; dg.z += s4.z; dg.w += s4.w;
                }
                const float4 g4 = ld4g(G + off);
                if (relu) {
                    dg.x = g4.x > 0.f ? dg.x : 0.f; dg.y = g4.y > 0.f ? dg.y : 0.f;
                    dg.z = g4.z > 0.f ? dg.z : 0.f; dg.w = g4.w > 0.f ? dg.w : 0.f;
                }
                const float rinv = rs[i];
                dn.x = dg.x * rinv; dn.y = dg.y * rinv; dn.z = dg.z * rinv; dn.w = dg.w * rinv;
                *reinterpret_cast<float4*>(dE + off) = dn;
                drp = -(dn.x * g4.x + dn.y * g4.y + dn.z * g4.z + dn.w * g4.w);
                zl = ld4g(Z + off);
            }
            *reinterpret_cast<float4*>(dNs + i * LDN + c0) = dn;
            *reinterpret_cast<float4*>(Ts + i * LDN + c0) = zl;
#pragma unroll
            for (int o = CG / 2; o > 0; o >>= 1) drp += __shfl_xor_sync(0xffffffffu, drp, o);
            if (cg == 0 && i < n) drs[i] += drp;
        }
        __syncthreads();
        // (c) dA += dN_l Z_l^T  (+ dr on the last processed sub-layer)
        for (int u = warp; u < MT * MT; u += SM_WARPS) {
            const int mt = u / MT, jt = u - mt * MT;
            float c[2][4];
            zero_frag<2>(c);
            const float* da = dNs + (16 * mt) * LDN;
            const float* zb = Ts + (16 * jt) * LDN;
            warp_gemm<2, true>(c, GD / 8, da, LDN, zb, LDN);
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int i = 16 * mt + g + 8 * half;
                if (i >= n) continue;
                const float dr = (l == 0) ? drs[i] : 0.f;
#pragma unroll
                for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int j = 16 * jt + 8 * nt + 2 * t + e;
                        if (j >= n) continue;
                        float* p = dAb + static_cast<size_t>(i) * n + j;
                        float val = c[nt][2 * half + e] + dr;
                        if (l != layers - 1) val += *p;
                        *p = val;
                    }
            }
        }
        __syncthreads();
        // (b) dZ_l = A^T dN_l  -> Ts (for the dense-connect push-down) and global
        for (int u = warp; u < MT * NG; u += SM_WARPS) {
            const int jt = u / NG, ng = u - jt * NG;
            float c[4][4];
            zero_frag<4>(c);
            const float* at = Ats + (16 * jt) * LDA;
            const float* db = dNs + 32 * ng;
            warp_gemm<4, false>(c, NP / 8, at, LDA, db, LDN);
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int j = 16 * jt + g + 8 * half;
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) {
                    const int col = 32 * ng + 8 * nt + 2 * t;
                    const float2 v = make_float2(c[nt][2 * half], c[nt][2 * half + 1]);
                    *reinterpret_cast<float2*>(Ts + j * LDN + col) = v;
                    if (j < n)
                        *reinterpret_cast<float2*>(dZ + static_cast<size_t>(node0 + j) * HD + colbase + col) = v;
                }
            }
        }
        __syncthreads();
        // push dZ_l through the dense connection: dG_m[j][c'] += sum_c dZ_l[j][c] * Wn_l[128 + m*GD + c'][c]
        for (int u = warp; u < l * MT * NG; u += SM_WARPS) {
            const int m = u / (MT * NG), rem = u - m * (MT * NG);
            const int jt = rem / NG, ng = rem - jt * NG;
            float c[4][4];
            zero_frag<4>(c);
            const float* ta = Ts + (16 * jt) * LDN;
            const float* wb = wsrc + static_cast<size_t>(m * GD + 32 * ng) * GD;
            warp_gemm<4, true>(c, GD / 8, ta, LDN, wb, GD);
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int j = 16 * jt + g + 8 * half;
                if (j >= n) continue;
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) {
                    const int col = 32 * ng + 8 * nt + 2 * t;
                    float* p = dZ + static_cast<size_t>(node0 + j) * HD + static_cast<size_t>(h) * S + m * GD + col;
                    float2 v = make_float2(c[nt][2 * half], c[nt][2 * half + 1]);
                    if (l != layers - 1) {
                        const float2 cur = *reinterpret_cast<const float2*>(p);
                        v.x += cur.x; v.y += cur.y;
                    }
                    *reinterpret_cast<float2*>(p) = v;
                }
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
static size_t fwd_mma_smem(int n, int layers, int gd) {
    const int np = (n + 15) & ~15, ki = (layers - 1) * gd;
    return (static_cast<size_t>(np) * (np + 4) + static_cast<size_t>(np) * (gd + 8) +
            static_cast<size_t>(np) * (ki + 4) + np) * sizeof(float);
}
static size_t bwd_mma_smem(int n, int layers, int gd) {
    const int np = (n + 15) & ~15;
    (void)layers;
    return (static_cast<size_t>(np) * (np + 4) + 2 * static_cast<size_t>(np) * (gd + 12) + 2 * np) * sizeof(float);
}

bool stack_mma_usable(const gcgcn_batch* bt, int layers, int slab) {
    if (layers < 1 || slab % layers != 0) return false;
    const int gd = slab / layers;
    return bt->max_nodes <= 64 && (gd == 32 || gd == 64);
}

int launch_stack_fwd_mma(const gcgcn_batch* bt, int heads, int layers, int slab, int flags, const float* A,
                         float* Z, const float* E, const float* Winner, const float* keep, const float* x,
                         float* G, float* F, cudaStream_t st) {
    const int gd = slab / layers;
    const long long* pp = reinterpret_cast<const long long*>(bt->pair_ptr);
    GCGCN_TRY(set_smem(stack_fwd_mma_kernel<64>, fwd_mma_smem(64, layers, 64), "stack_fwd_mma"));
    GCGCN_TRY(set_smem(stack_fwd_mma_kernel<32>, fwd_mma_smem(64, layers, 32), "stack_fwd_mma"));
    return for_each_size_class(bt, [&](int count, int first, int nmax, const int* order) -> int {
        const size_t smem = fwd_mma_smem(nmax, layers, gd);
        dim3 grid(count, heads);
        if (gd == 64)
            stack_fwd_mma_kernel<64><<<grid, SM_THREADS, smem, st>>>(bt->node_ptr, pp, A, Z, E, Winner, keep, x, G, F,
                                                                     layers, heads, flags, bt->total_pairs, order, first);
        else
            stack_fwd_mma_kernel<32><<<grid, SM_THREADS, smem, st>>>(bt->node_ptr, pp, A, Z, E, Winner, keep, x, G, F,
                                                                     layers, heads, flags, bt->total_pairs, order, first);
        GCGCN_CHECK_LAUNCH("gcn_stack_fwd_mma");
        return GCGCN_OK;
    });
}

int launch_stack_bwd_mma(const gcgcn_batch* bt, int heads, int layers, int slab, int flags, const float* A,
                         const float* Z, const float* G, const float* Winner, const float* keep, const float* dF,
                         float* dZ, float* dE, float* dA, cudaStream_t st) {
    const int gd = slab / layers;
    const long long* pp = reinterpret_cast<const long long*>(bt->pair_ptr);
    GCGCN_TRY(set_smem(stack_bwd_mma_kernel<64>, bwd_mma_smem(64, layers, 64), "stack_bwd_mma"));
    GCGCN_TRY(set_smem(stack_bwd_mma_kernel<32>, bwd_mma_smem(64, layers, 32), "stack_bwd_mma"));
    return for_each_size_class(bt, [&](int count, int first, int nmax, const int* order) -> int {
        const size_t smem = bwd_mma_smem(nmax, layers, gd);
        dim3 grid(count, heads);
        if (gd == 64)
            stack_bwd_mma_kernel<64><<<grid, SM_THREADS, smem, st>>>(bt->node_ptr, pp, A, Z, G, Winner, keep, dF, dZ, dE,
                                                                     dA, layers, heads, flags, bt->total_pairs, order, first);
        else
            stack_bwd_mma_kernel<32><<<grid, SM_THREADS, smem, st>>>(bt->node_ptr, pp, A, Z, G, Winner, keep, dF, dZ, dE,
                                                                     dA, layers, heads, flags, bt->total_pairs, order, first);
        GCGCN_CHECK_LAUNCH("gcn_stack_bwd_mma");
        return GCGCN_OK;
    });
}

}  // namespace gcgcn
