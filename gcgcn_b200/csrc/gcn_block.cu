// CAGGC / MAGGC graph-block kernels for DocRED-sized graphs (n <= 64): one CTA per (document, head).
//
// This is the block form of the dense-connected GraphConv stack (G:63-80, G:97-120) with the attention
// step that feeds it fused in:
//   forward   P_h = softmax(q_h q_h^T / sqrt(d_h))            (MHA, G:133-142; key = query projection)
//             or the given attention map (CAGGC: GATAttention's map from the edge pass)
//             for l < L:  Z_l = Zx_l + g_{<l} Winner_l ;  g_l = relu((E_l + P Z_l) / r) ;  F_l = g_l + x_l
//   backward  dE_l = dN_l = relu'(g_l) dF_l / r ;  dA += dN_l Z_l^T ;  dZ_l = P^T dN_l ;  dense-connect push-down ;
//             then, without leaving the CTA, the softmax backward dS = P (dA - rowsum(dA P)) and either
//             dq_h = scale (dS + dS^T) q_h  (MHA)  or dS itself (GAT; the edge pass consumes it).
//
// Why these kernels replaced a plain per-document mma.sync stack kernel, and what ncu said at each step:
//   1. the first kernel was latency bound (long-scoreboard stalls on five dependent global round trips per
//      CTA): here the per-sub-layer projection tiles arrive by cp.async into a two-deep ring and the epilogue
//      operands are loaded ahead of the MMA loop that precedes their use; the attention map and its gradient
//      never leave shared memory between sub-layers; the softmax, its backward and the dq reduction ride
//      along instead of being three more passes over [H][sum n^2] arrays in HBM;
//   2. then it was instruction bound with HMMA at 13 % of the issued instructions (fragment loads as scalar LDS,
//      the hi/lo split redone per fragment use, run-time strides): operands are split once into hi/lo planes,
//      fragments come from ldmatrix, and every size class (16/32/48/64 rows) is its own instantiation so that
//      strides are immediates and the tile loops unroll;
//   3. then the L1/shared pipe was the limiter (80-90 %): one row tile x several column tiles per warp (the
//      1 KB row fragment is read once per 2-4 cheap column fragments) and the dense-connect weights are read in
//      MMA-fragment order (one 128-byte line per fragment register instead of 4-8 sectors).
//
// All small matrix products run on the tensor cores (mma.sync m16n8k8 TF32, 3xTF32 split, see
// mma_tf32.cuh).  Block configuration only: slab = in_dim = 128, ReLU + residual, no dropout masks
// (keep masks passed in as tensors take the row-tiled kernels of gcn_stack_tiled.cu).
#include "common.cuh"
#include "mma_tf32.cuh"

namespace gcgcn {

constexpr int BK_THREADS = 256;
constexpr int BK_WARPS = BK_THREADS / WARP;

enum { BK_OUT_DA = 0, BK_OUT_DS = 1, BK_OUT_DQ = 2 };

__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gsrc) {
    const uint32_t d = static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst));
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// ---- operand planes and fragment loads -----------------------------------------------------
// Every MMA operand that several warps read lives in shared memory already split into a TF32-exact "hi"
// plane and an fp32 "lo = x - hi" plane (the split is paid once per element, not once per fragment use),
// with rows of stride == 4 (mod 8) words so that ldmatrix -- whose 8x8 b16 tile is an 8x4 tile of 32-bit
// words, exactly one m16n8k8 TF32 fragment register per lane -- is bank-conflict free.
__device__ __forceinline__ uint32_t s_addr(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void ldsm4(uint32_t (&r)[4], const float* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(s_addr(p))
                 : "memory");
}
__device__ __forceinline__ void split_f(float x, float& hi, float& lo) {
    hi = __uint_as_float(__float_as_uint(x) & 0xffffe000u);
    lo = x - hi;
}
__device__ __forceinline__ void split_f4(const float4 v, float4& hi, float4& lo) {
    split_f(v.x, hi.x, lo.x); split_f(v.y, hi.y, lo.y); split_f(v.z, hi.z, lo.z); split_f(v.w, hi.w, lo.w);
}
// c += a b  with  a = ah + al, b = bh + bl  (3xTF32: the lo*lo term is below fp32 resolution)
__device__ __forceinline__ void mma3(float (&c)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4], uint32_t bh0,
                                     uint32_t bh1, uint32_t bl0, uint32_t bl1) {
    const uint32_t bh[2] = {bh0, bh1}, bl[2] = {bl0, bl1};
    mma_tf32(c, al, bh);
    mma_tf32(c, ah, bl);
    mma_tf32(c, ah, bh);
}
__device__ __forceinline__ void mma3f(float (&c)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4], float b0,
                                      float b1) {
    float h0, l0, h1, l1;
    split_f(b0, h0, l0);
    split_f(b1, h1, l1);
    mma3(c, ah, al, __float_as_uint(h0), __float_as_uint(h1), __float_as_uint(l0), __float_as_uint(l1));
}
__device__ __forceinline__ float group8_sum(float v) {
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    return v;
}
__device__ __forceinline__ float group8_max(float v) {
    v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
    v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
    v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 4));
    return v;
}

// Warp tiling of a [16 MT] x [8 NT] product: each warp takes one row tile and NTW column tiles, NTW the smallest
// power of two that fits all MT * NT / NTW units into the 8 warps.
__host__ __device__ constexpr int col_tiles_per_warp(int mt, int nt) {
    int w = 1;
    while (mt * (nt / w) > BK_WARPS && w < nt) w *= 2;
    return w;
}

// ---- dense-connect weights in MMA-fragment order ----------------------------------------------------
// The B fragments of the dense-connect products come straight from global memory (16-24 KB per head, L1/L2
// resident).  Read from the row-major Winner block, one fragment load touches 4-8 different 32-byte sectors;
// re-ordered once per call so that the 32 lanes of a fragment register are contiguous -- and already split
// into hi/lo -- it is one 128-byte line per register.
//   forward  (B(k, n) = W_l[k][n]):            Wf[h][l][ks][nt][q][lane],      k = 8 ks + t + 4 (q & 1), n = 8 nt + g
//   backward (B(k, n) = W_l[m gd + n][k]):     Wb[h][l][m][ks][nt][q][lane],   k = 8 ks + t + 4 (q & 1), n = 8 nt + g
// q = {hi b0, hi b1, lo b0, lo b1}, lane = 4 g + t.  Both arrays hold heads * layers * KI * gd * 2 floats.
size_t block_frag_floats(int heads, int layers) {
    const int gd = D / layers, ki = (layers - 1) * gd;
    return 2 * static_cast<size_t>(heads) * layers * ki * gd * 2;      // Wf then Wb
}

__global__ void __launch_bounds__(256)
winner_frag_kernel(const float* __restrict__ Winner, int layers, int gd, float* __restrict__ Wf, float* __restrict__ Wb) {
    const int hl = blockIdx.x, l = hl % layers;
    const int ki = (layers - 1) * gd, nt_n = gd / 8;
    const size_t per = static_cast<size_t>(ki) * gd * 2;
    const float* W = Winner + static_cast<size_t>(hl) * D * gd;           // [128][gd] block of GraphConv (h, l)
    for (int idx = blockIdx.y * blockDim.x + threadIdx.x; idx < static_cast<int>(per); idx += gridDim.y * blockDim.x) {
        const int lane = idx & 31, q = (idx >> 5) & 3, g = lane >> 2, t = lane & 3;
        const int rest = idx >> 7;                                        // (ks, nt) forward; (m, ks, nt) backward
        const int nt = rest % nt_n;
        {   // forward order
            const int ks = rest / nt_n;
            const int k = 8 * ks + t + 4 * (q & 1), n = 8 * nt + g;
            const float v = k < l * gd ? W[static_cast<size_t>(k) * gd + n] : 0.f;
            const float hi = __uint_as_float(__float_as_uint(v) & 0xffffe000u);
            Wf[hl * per + idx] = (q & 2) ? v - hi : hi;
        }
        {   // backward order
            const int ks = (rest / nt_n) % nt_n, m = rest / (nt_n * nt_n);
            const int k = 8 * ks + t + 4 * (q & 1), row = m * gd + 8 * nt + g;
            const float v = m < l ? W[static_cast<size_t>(row) * gd + k] : 0.f;
            const float hi = __uint_as_float(__float_as_uint(v) & 0xffffe000u);
            Wb[hl * per + idx] = (q & 2) ? v - hi : hi;
        }
    }
}

// Materialises one dropout stream (tests compare the in-kernel dropout with the keep-mask-in route).
__global__ void __launch_bounds__(256)
dropout_mask_kernel(unsigned long long seed, uint32_t stream, uint32_t thr, float inv, long long count, float* __restrict__ out) {
    const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx < count) out[idx] = thr != 0u ? drop_keep(seed, stream, idx, thr, inv) : 1.f;
}
int launch_dropout_mask(unsigned long long seed, uint32_t stream, uint32_t thr, float inv, long long count, float* out,
                        cudaStream_t st) {
    if (count <= 0) return GCGCN_OK;
    dropout_mask_kernel<<<ceil_div(count, 256), 256, 0, st>>>(seed, stream, thr, inv, count, out);
    GCGCN_CHECK_LAUNCH("dropout_mask");
    return GCGCN_OK;
}

// Per-lane geometry shared by both kernels.
//   ldmatrix A fragment (16 rows x 8 k): lane supplies row a_row, k offset a_col of the tile
//   ldmatrix B fragment, operand stored [n][k] (hi and lo planes in one x4): row b_row, k offset b_col, plane b_lo
//   row-wise passes: 8 lanes per attention row (4 rows per warp, 32 per CTA pass), lane l8 takes columns l8 + 8r
struct LaneGeo {
    int warp, lane, g, t, a_row, a_col, b_row, b_col, b_lo, l8, rsub;
    __device__ __forceinline__ LaneGeo() {
        warp = threadIdx.x >> 5; lane = threadIdx.x & 31;
        g = lane >> 2; t = lane & 3;
        a_row = (lane & 7) + ((lane >> 3) & 1) * 8; a_col = (lane >> 4) * 4;
        b_row = lane & 7; b_col = ((lane >> 3) & 1) * 4; b_lo = lane >> 4;
        l8 = lane & 7; rsub = warp * 4 + (lane >> 3);
    }
};

// ---------------------------------------------------------------------------------------------
// DH = 0: attention map given in A.  DH > 0: MHA scores from the head slice of q (width DH); P is written.
// MTC = size class: every document of the launch is padded to NP = 16 MTC rows (compile-time strides, fully
// unrolled tile loops -- with run-time strides the integer address arithmetic outweighed the MMAs 4:1).
template <int GD, int DH, int MTC>
__global__ void __launch_bounds__(BK_THREADS, MTC <= 2 ? 4 : 3)
block_fwd_kernel(const int* __restrict__ node_ptr, const long long* __restrict__ pair_ptr,
                 const float* __restrict__ A, const float* __restrict__ q, float* __restrict__ P,
                 float* __restrict__ Z, const float* __restrict__ E, const float* __restrict__ Wf,
                 const float* __restrict__ x, float* __restrict__ G, float* __restrict__ F, int heads,
                 long long total_pairs, const int* __restrict__ doc_order, int first, float scale, const BlockDrop drop) {
    extern __shared__ __align__(16) float smem[];
    const int b = doc_order != nullptr ? doc_order[first + blockIdx.x] : blockIdx.x;
    const int h = blockIdx.y;
    const int node0 = node_ptr[b];
    const int n = node_ptr[b + 1] - node0;
    if (n == 0) return;
    constexpr int S = D, layers = D / GD, LDZ = GD + 8, CG = GD / 4, DHH = DH > 0 ? DH : 8;
    constexpr int NTW = col_tiles_per_warp(MTC, GD / 8), NG = (GD / 8) / NTW, UNITS = MTC * NG;
    constexpr int NP = 16 * MTC, MT = MTC, NT8 = 2 * MTC, LDA = NP + 4, KI = (layers - 1) * GD, LDG = KI + 4;
    const int HD = DH > 0 ? (D / DHH) * S : heads * S;

    float* Ahi = smem;                 // [NP][LDA]    attention map, zero padded, hi plane
    float* Alo = Ahi + NP * LDA;       // [NP][LDA]    lo plane (scratch for the raw scores before the softmax)
    float* Zs0 = Alo + NP * LDA;       // [2][NP][LDZ] ring of projection tiles Zx_l (-> Z_l in place), fp32
    float* Ghi = Zs0 + 2 * NP * LDZ;   // [NP][LDG]    g_0 .. g_{L-2}, hi plane
    float* Glo = Ghi + NP * LDG;       // [NP][LDG]    lo plane
    float* rs = Glo + NP * LDG;        // [NP]         reciprocal row normalisers

    const int tid = threadIdx.x;
    const LaneGeo L;
    const long long abase = static_cast<long long>(h) * total_pairs + pair_ptr[b];
    const size_t hbase = static_cast<size_t>(node0) * HD + h * S;       // + i*HD + l*GD + col  (32-bit offsets)
    const float* zsrc = Z + hbase;
    const float* Eb = E + hbase;
    float* Gb = G + hbase;
    float* Fb = F + hbase;
    const float* xb = x + static_cast<size_t>(node0) * S;

    auto issue_z = [&](int l) {        // rows < n of the x-part projection of sub-layer l -> ring slot l & 1
        float* dst = Zs0 + (l & 1) * NP * LDZ;
        const float* src = zsrc + l * GD;
        for (int idx = tid; idx < n * CG; idx += BK_THREADS) {
            const int i = idx / CG, c4 = (idx - i * CG) * 4;
            cp_async16(dst + i * LDZ + c4, src + i * HD + c4);
        }
    };
    issue_z(0);
    cp_async_commit();
    if (layers > 1) issue_z(1);
    cp_async_commit();
    // padding rows (never touched by cp.async or the epilogues) must be exact zeros: they are MMA operands
    for (int idx = tid; idx < (NP - n) * LDZ; idx += BK_THREADS) {
        Zs0[n * LDZ + idx] = 0.f;
        Zs0[NP * LDZ + n * LDZ + idx] = 0.f;
    }

    if (DH > 0) {
        // ---- MHA scores on the tensor cores: S = scale q_h q_h^T (fp32 via 3xTF32) -> Alo ----
        constexpr int LQ = DHH + 4, Q4 = DHH / 4;
        float* qh = Ghi;               // [NP][LQ] hi / lo planes of the head slice of q; dead before g_0 exists
        float* ql = Glo;
        for (int idx = tid; idx < NP * Q4; idx += BK_THREADS) {
            const int j = idx / Q4, k4 = (idx - j * Q4) * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f), hi, lo;
            if (j < n) v = ld4g(q + static_cast<size_t>(node0 + j) * D + h * DHH + k4);
            split_f4(v, hi, lo);
            *reinterpret_cast<float4*>(qh + j * LQ + k4) = hi;
            *reinterpret_cast<float4*>(ql + j * LQ + k4) = lo;
        }
        __syncthreads();
        for (int u = L.warp; u < MT * NT8; u += BK_WARPS) {
            const int mt = u / NT8, nt = u - mt * NT8;
            float c[4] = {0.f, 0.f, 0.f, 0.f};
            const float* pa = qh + (16 * mt + L.a_row) * LQ + L.a_col;
            const float* pb = (L.b_lo ? ql : qh) + (8 * nt + L.b_row) * LQ + L.b_col;
#pragma unroll
            for (int k0 = 0; k0 < DHH; k0 += 8) {
                uint32_t ah[4], al[4], bb[4];
                ldsm4(ah, pa + k0);
                ldsm4(al, pa + NP * LDG + k0);
                ldsm4(bb, pb + k0);
                mma3(c, ah, al, bb[0], bb[1], bb[2], bb[3]);
            }
            float* srow = Alo + (16 * mt + L.g) * LDA + 8 * nt + 2 * L.t;
            *reinterpret_cast<float2*>(srow) = make_float2(c[0] * scale, c[1] * scale);
            *reinterpret_cast<float2*>(srow + 8 * LDA) = make_float2(c[2] * scale, c[3] * scale);
        }
        __syncthreads();
    }
    for (int idx = tid; idx < (NP - n) * LDG; idx += BK_THREADS) {   // padding rows of the g planes (q is dead now)
        Ghi[n * LDG + idx] = 0.f;
        Glo[n * LDG + idx] = 0.f;
    }
    // ---- attention rows: softmax (MHA) or load (given), hi/lo planes, reciprocal row normalisers (G:47-49) ----
#pragma unroll
    for (int r0 = 0; r0 < NP; r0 += 32) {
        const int i = r0 + L.rsub;
        if (i >= NP) continue;         // warp-uniform: a warp owns 4 consecutive rows, NP is a multiple of 16
        const bool rv = i < n;
        float v[8];
        float m = -INFINITY;
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int j = L.l8 + 8 * r;
            v[r] = -INFINITY;
            if (r < NT8 && rv && j < n) {
                v[r] = DH > 0 ? Alo[i * LDA + j] : A[abase + static_cast<long long>(i) * n + j];
                m = fmaxf(m, v[r]);
            }
        }
        float inv = 1.f;
        if (DH > 0) {
            m = group8_max(m);
            float z = 0.f;
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                v[r] = (v[r] == -INFINITY) ? 0.f : __expf(v[r] - m);
                z += v[r];
            }
            z = group8_sum(z);
            inv = rv ? 1.0f / z : 0.f;
        }
        float sum = 0.f;
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int j = L.l8 + 8 * r;
            if (r < NT8) {
                float p = 0.f;
                if (rv && j < n) {
                    p = v[r] * inv;
                    const long long pidx = abase + static_cast<long long>(i) * n + j;
                    if (DH > 0) P[pidx] = p;                   // softmax output, saved for backward (pre-dropout)
                    if (drop.thr_att != 0u) p *= drop_keep(drop.seed, drop.s_att, pidx, drop.thr_att, drop.inv_att);   // G:141, G:166
                }
                float hi, lo;
                split_f(p, hi, lo);
                Ahi[i * LDA + j] = hi;
                Alo[i * LDA + j] = lo;
                sum += p;
            }
        }
        sum = group8_sum(sum);
        if (L.l8 == 0) rs[i] = 1.0f / (sum + (sum == 0.f ? 1.f : 0.f));
    }

#pragma unroll
    for (int l = 0; l < layers; ++l) {
        float* Zs = Zs0 + (l & 1) * NP * LDZ;
        const int kin = l * GD;
        cp_async_wait<1>();            // this thread's copies of tile l have landed ...
        __syncthreads();               // ... and everyone's; also publishes the attention planes / g_{l-1}
        // warp -> unit (row tile mt, group ng of NTW column tiles): the expensive fragment (16 x 8 hi+lo of the
        // row operand, 8 shared-memory wavefronts) is loaded once per NTW cheap column fragments
        const int mt = L.warp / NG, ng = L.warp - mt * NG;
        const bool busy = L.warp < UNITS;
        const int col0 = 8 * NTW * ng;                                 // first column of this warp's tile
        float c[NTW][4];
        float* zc = Zs + (16 * mt + L.g) * LDZ + col0 + 2 * L.t;      // this lane's C-fragment corner in the tile
        if (l > 0) {
            // Z_l += g_{<l} Winner_l   (dense connection, row-local in the reference: G:72-73)
            if (busy) {
                // fragment-ordered hi/lo weights: [ks][nt][4][32] floats per (head, sub-layer)
                const float* wb = Wf + (static_cast<size_t>(h) * layers + l) * (KI * GD * 2) + (col0 / 8) * 128 + L.lane;
#pragma unroll
                for (int nt = 0; nt < NTW; ++nt) {
                    const float2 lo2 = *reinterpret_cast<const float2*>(zc + 8 * nt);
                    const float2 hi2 = *reinterpret_cast<const float2*>(zc + 8 * LDZ + 8 * nt);
                    c[nt][0] = lo2.x; c[nt][1] = lo2.y; c[nt][2] = hi2.x; c[nt][3] = hi2.y;
                }
                const float* pa = Ghi + (16 * mt + L.a_row) * LDG + L.a_col;
#pragma unroll 2
                for (int k0 = 0; k0 < kin; k0 += 8) {
                    uint32_t ah[4], al[4];
                    ldsm4(ah, pa + k0);
                    ldsm4(al, pa + NP * LDG + k0);
#pragma unroll
                    for (int nt = 0; nt < NTW; ++nt) {
                        const float* f = wb + (k0 / 8) * (GD / 8) * 128 + nt * 128;
                        mma3(c[nt], ah, al, __float_as_uint(__ldg(f)), __float_as_uint(__ldg(f + 32)),
                             __float_as_uint(__ldg(f + 64)), __float_as_uint(__ldg(f + 96)));
                    }
                }
#pragma unroll
                for (int nt = 0; nt < NTW; ++nt) {
                    *reinterpret_cast<float2*>(zc + 8 * nt) = make_float2(c[nt][0], c[nt][1]);
                    *reinterpret_cast<float2*>(zc + 8 * LDZ + 8 * nt) = make_float2(c[nt][2], c[nt][3]);
                }
            }
            __syncthreads();
            for (int idx = tid; idx < n * CG; idx += BK_THREADS) {       // final Z_l, saved for backward
                const int i = idx / CG, c4 = (idx - i * CG) * 4;
                *reinterpret_cast<float4*>(Z + hbase + (i * HD + kin + c4)) =
                    *reinterpret_cast<const float4*>(Zs + i * LDZ + c4);
            }
        }
        // out = (E + P Z_l) / r ; g_l = relu(out) ; F_l = g_l + x_l
        if (busy) {
            // epilogue operands first: their latency hides behind the MMA loop
            float2 e2[2][NTW], x2[2][NTW];
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int i = 16 * mt + L.g + 8 * half;
#pragma unroll
                for (int nt = 0; nt < NTW; ++nt) {
                    e2[half][nt] = make_float2(0.f, 0.f);
                    x2[half][nt] = make_float2(0.f, 0.f);
                    if (i < n) {
                        const int col = col0 + 8 * nt + 2 * L.t;
                        e2[half][nt] = ld2g(Eb + (i * HD + kin + col));
                        x2[half][nt] = ld2g(xb + (i * S + kin + col));
                    }
                }
            }
#pragma unroll
            for (int nt = 0; nt < NTW; ++nt) { c[nt][0] = 0.f; c[nt][1] = 0.f; c[nt][2] = 0.f; c[nt][3] = 0.f; }
            const float* pa = Ahi + (16 * mt + L.a_row) * LDA + L.a_col;
            const float* zb = Zs + L.t * LDZ + col0 + L.g;
#pragma unroll
            for (int k0 = 0; k0 < NP; k0 += 8) {
                uint32_t ah[4], al[4];
                ldsm4(ah, pa + k0);
                ldsm4(al, pa + NP * LDA + k0);
#pragma unroll
                for (int nt = 0; nt < NTW; ++nt) mma3f(c[nt], ah, al, zb[k0 * LDZ + 8 * nt], zb[(k0 + 4) * LDZ + 8 * nt]);
            }
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int i = 16 * mt + L.g + 8 * half;
                if (i >= n) continue;
                const float rinv = rs[i];
#pragma unroll
                for (int nt = 0; nt < NTW; ++nt) {
                    const int col = col0 + 8 * nt + 2 * L.t;
                    const int off = i * HD + kin + col;
                    float2 o;
                    o.x = fmaxf((e2[half][nt].x + c[nt][2 * half]) * rinv, 0.f);
                    o.y = fmaxf((e2[half][nt].y + c[nt][2 * half + 1]) * rinv, 0.f);
                    *reinterpret_cast<float2*>(Gb + off) = o;
                    float2 f = o;                                // dropout hits only the output copy (G:72-74)
                    if (drop.thr_gcn != 0u) {
                        const float2 k2 = drop_keep2(drop.seed, drop.s_gcn, hbase + off, drop.thr_gcn, drop.inv_gcn);
                        f.x *= k2.x; f.y *= k2.y;
                    }
                    *reinterpret_cast<float2*>(Fb + off) = make_float2(f.x + x2[half][nt].x, f.y + x2[half][nt].y);
                    if (l < layers - 1) {
                        float2 hi, lo;
                        split_f(o.x, hi.x, lo.x);
                        split_f(o.y, hi.y, lo.y);
                        *reinterpret_cast<float2*>(Ghi + i * LDG + kin + col) = hi;
                        *reinterpret_cast<float2*>(Glo + i * LDG + kin + col) = lo;
                    }
                }
            }
        }
        __syncthreads();               // ring slot l & 1 is free again
        if (l + 2 < layers) issue_z(l + 2);
        cp_async_commit();             // (possibly empty) keeps "all but the newest group" == tile l+1
    }
    cp_async_wait<0>();
}

// ---------------------------------------------------------------------------------------------
// OUT = BK_OUT_DA: dA (head-major, like A) is written and the softmax backward is left to the caller.
// OUT = BK_OUT_DS: A is a softmax output; dS = A (dA - rowsum(dA A)) is written instead (GAT, one head).
// OUT = BK_OUT_DQ: as DS, then dq_h = scale (dS + dS^T) q_h is written to the head slice of dq [rows][128].
template <int GD, int DH, int OUT, int MTC>
__global__ void __launch_bounds__(BK_THREADS, MTC <= 2 ? 4 : 3)
block_bwd_kernel(const int* __restrict__ node_ptr, const long long* __restrict__ pair_ptr,
                 const float* __restrict__ A, const float* __restrict__ q, const float* __restrict__ Z,
                 const float* __restrict__ G, const float* __restrict__ Wb, const float* __restrict__ dF,
                 float* __restrict__ dZ, float* __restrict__ dE, float* __restrict__ dOut, int heads,
                 long long total_pairs, const int* __restrict__ doc_order, int first, float scale, const BlockDrop drop) {
    extern __shared__ __align__(16) float smem[];
    const int b = doc_order != nullptr ? doc_order[first + blockIdx.x] : blockIdx.x;
    const int h = blockIdx.y;
    const int node0 = node_ptr[b];
    const int n = node_ptr[b + 1] - node0;
    if (n == 0) return;
    constexpr int S = D, layers = D / GD, CG = GD / 4, RPP = BK_THREADS / CG;
    // dN / T planes [NP][LDN].  Sub-layer width 64: rows of exactly 64 words with the 16-byte chunk index XORed with
    // plane_mask(row) -- ldmatrix (8 rows x one chunk) and the B fragments of dZ = A^T dN (rows k0 + t, columns g,
    // read as scalars: ldmatrix cannot transpose 32-bit elements) are then both bank-conflict free; with the padded
    // row-major layout the latter were 2-way conflicted and made up a quarter of the kernel's shared-memory
    // wavefronts, on the pipe that bounds it (ncu: l1tex data pipe 71-88 %).  Width 32 keeps the padded layout (its
    // dq operands need the larger area).
    constexpr bool SWZ = (GD == 64);
    constexpr int LDN = SWZ ? GD : GD + 12;
    constexpr int DHH = DH > 0 ? DH : 8;
    constexpr int NTW = col_tiles_per_warp(MTC, GD / 8), NG = (GD / 8) / NTW, UNITS = MTC * NG;           // [NP] x [GD] products
    constexpr int NTW_C = MTC, NG_C = 2, UNITS_C = 2 * MTC;          // [NP] x [NP]: a row tile x half the columns per warp
    constexpr int NP = 16 * MTC, MT = MTC, NT8 = 2 * MTC, LDA = NP + 4, KI = (layers - 1) * GD, LDG = KI + 4;
    const int HD = DH > 0 ? (D / DHH) * S : heads * S;

    // Shared memory is what limits residency here, so: the attention map is one fp32 plane (its fragments are
    // split in registers), dA accumulates in registers across the sub-layers, and with two sub-layers the single
    // parked dense-connect gradient lives in the (then dead) dN hi plane.
    constexpr bool TWO = (layers == 2);
    float* AtS = smem;                 // [NP][LDA]  A transposed: AtS[j][i] = A[i][j], fp32
    float* dNh = AtS + NP * LDA;       // [NP][LDN]  dN_l = relu'(g_l) dG_l / r, hi / lo planes
    float* dNl = dNh + NP * LDN;
    float* Th = dNl + NP * LDN;        // [NP][LDN]  Z_l, then dZ_l, hi / lo planes
    float* Tl = Th + NP * LDN;
    float* rs = Tl + NP * LDN;         // [NP]
    float* drs = rs + NP;              // [NP]
    // dA / dS scratch of the final phase [NP][LDA]: the tail of the (dead) T planes, or its own region when the
    // head of the dN/T area is too small for the dq operands (sub-layer width 32)
    float* dAs = TWO ? Tl + NP * LDN - NP * LDA : drs + NP;
    float* dGs = TWO ? dNh : dAs + NP * LDA;      // [NP][LDG or LDN]  dense-connect gradient parked for sub-layers < l
    constexpr int LDP = TWO ? LDN : LDG;          // its row stride

    const int tid = threadIdx.x;
    const LaneGeo L;
    // word offset of (row, col) in a dN / T plane; mask = {0,2,4,6,1,3,5,7}[row & 7]
    auto pl = [](int row, int col) -> int {
        if (!SWZ) return row * LDN + col;
        const int mask = ((row & 3) << 1) | ((row >> 2) & 1);
        return row * LDN + ((((col >> 2) ^ mask) << 2) | (col & 3));
    };
    const long long abase = static_cast<long long>(h) * total_pairs + pair_ptr[b];
    const float* Ab = A + abase;
    const size_t hbase = static_cast<size_t>(node0) * HD + h * S;       // + i*HD + l*GD + col  (32-bit offsets)

#pragma unroll
    for (int r0 = 0; r0 < NP; r0 += 32) {
        const int i = r0 + L.rsub;
        if (i >= NP) continue;
        float sum = 0.f;
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int j = L.l8 + 8 * r;
            if (r < NT8) {
                float v = (i < n && j < n) ? Ab[i * n + j] : 0.f;
                if (drop.thr_att != 0u && i < n && j < n)       // A = P * keep, regenerated (Ab then holds the softmax output P)
                    v *= drop_keep(drop.seed, drop.s_att, abase + i * n + j, drop.thr_att, drop.inv_att);
                AtS[j * LDA + i] = v;
                sum += v;
            }
        }
        sum = group8_sum(sum);
        if (L.l8 == 0) { rs[i] = 1.0f / (sum + (sum == 0.f ? 1.f : 0.f)); drs[i] = 0.f; }
    }
    __syncthreads();

    const int cg = tid % CG, rg = tid / CG, c0 = cg * 4;
    float cA[NTW_C][4];
#pragma unroll
    for (int nt = 0; nt < NTW_C; ++nt) { cA[nt][0] = 0.f; cA[nt][1] = 0.f; cA[nt][2] = 0.f; cA[nt][3] = 0.f; }
#pragma unroll
    for (int l = layers - 1; l >= 0; --l) {
        const float* wsrc = Wb + (static_cast<size_t>(h) * layers + l) * (KI * GD * 2);   // [m][ks][nt][4][32]
        const bool first_layer = (l == layers - 1);
        // (a) row-local: dG_l -> dN_l (shared), dE_l (global), dr (shared); Z_l -> shared
#pragma unroll
        for (int i0 = 0; i0 < NP; i0 += RPP) {
            const int i = i0 + rg;
            if (NP % RPP != 0 && i >= NP) continue;        // warp-uniform (RPP rows = 2 or 4 per warp)
            float4 dn = make_float4(0.f, 0.f, 0.f, 0.f), zl = dn;
            float drp = 0.f;
            if (i < n) {
                const size_t off = hbase + (i * HD + l * GD + c0);
                float4 dg = ld4g(dF + off);
                const float4 g4 = ld4g(G + off);
                zl = ld4g(Z + off);
                if (drop.thr_gcn != 0u) {
                    const float2 k01 = drop_keep2(drop.seed, drop.s_gcn, off, drop.thr_gcn, drop.inv_gcn);
                    const float2 k23 = drop_keep2(drop.seed, drop.s_gcn, off + 2, drop.thr_gcn, drop.inv_gcn);
                    dg.x *= k01.x; dg.y *= k01.y; dg.z *= k23.x; dg.w *= k23.y;
                }
                if (!first_layer) {
                    const float4 s4 = *reinterpret_cast<const float4*>(dGs + (TWO ? pl(i, l * GD + c0) : i * LDP + l * GD + c0));
                    dg.x += s4.x; dg.y += s4.y; dg.z += s4.z; dg.w += s4.w;
                }
                dg.x = g4.x > 0.f ? dg.x : 0.f; dg.y = g4.y > 0.f ? dg.y : 0.f;
                dg.z = g4.z > 0.f ? dg.z : 0.f; dg.w = g4.w > 0.f ? dg.w : 0.f;
                const float rinv = rs[i];
                dn.x = dg.x * rinv; dn.y = dg.y * rinv; dn.z = dg.z * rinv; dn.w = dg.w * rinv;
                *reinterpret_cast<float4*>(dE + off) = dn;
                drp = -(dn.x * g4.x + dn.y * g4.y + dn.z * g4.z + dn.w * g4.w);
            }
            float4 hi, lo;
            split_f4(dn, hi, lo);
            *reinterpret_cast<float4*>(dNh + pl(i, c0)) = hi;
            *reinterpret_cast<float4*>(dNl + pl(i, c0)) = lo;
            split_f4(zl, hi, lo);
            *reinterpret_cast<float4*>(Th + pl(i, c0)) = hi;
            *reinterpret_cast<float4*>(Tl + pl(i, c0)) = lo;
#pragma unroll
            for (int o = CG / 2; o > 0; o >>= 1) drp += __shfl_xor_sync(0xffffffffu, drp, o);
            if (cg == 0 && i < n) drs[i] += drp;
        }
        __syncthreads();
        // (c) dA += dN_l Z_l^T      (both operands K-contiguous: ldmatrix on either side; accumulators live in
        //     registers across the sub-layers)
        if (L.warp < UNITS_C) {
            const int mt = L.warp / NG_C, jg = L.warp - mt * NG_C;
            float (&c)[NTW_C][4] = cA;
            const int arow = 16 * mt + L.a_row, brow = 8 * NTW_C * jg + L.b_row;     // (+ 8 nt: same row & 7, same mask)
            const float* pb = L.b_lo ? Tl : Th;
#pragma unroll
            for (int k0 = 0; k0 < GD; k0 += 8) {
                uint32_t ah[4], al[4];
                const float* pa = dNh + pl(arow, L.a_col + k0);
                ldsm4(ah, pa);
                ldsm4(al, pa + NP * LDN);
                const int boff = pl(brow, L.b_col + k0);
#pragma unroll
                for (int nt = 0; nt < NTW_C; ++nt) {
                    uint32_t bb[4];
                    ldsm4(bb, pb + boff + 8 * nt * LDN);
                    mma3(c[nt], ah, al, bb[0], bb[1], bb[2], bb[3]);
                }
            }
        }
        // (b) dZ_l = A^T dN_l  -> T planes (for the dense-connect push-down) and global
        const int jt = L.warp / NG, ng = L.warp - jt * NG;
        const bool busy = L.warp < UNITS;
        const int col0 = 8 * NTW * ng;
        {
            float c[NTW][4];
#pragma unroll
            for (int nt = 0; nt < NTW; ++nt) { c[nt][0] = 0.f; c[nt][1] = 0.f; c[nt][2] = 0.f; c[nt][3] = 0.f; }
            if (busy) {
                const float* pa = AtS + (16 * jt + L.a_row) * LDA + L.a_col;
#pragma unroll
                for (int k0 = 0; k0 < NP; k0 += 8) {
                    uint32_t ah[4], al[4];
                    ldsm4(ah, pa + k0);
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        float hi, lo;
                        split_f(__uint_as_float(ah[e]), hi, lo);
                        ah[e] = __float_as_uint(hi);
                        al[e] = __float_as_uint(lo);
                    }
#pragma unroll
                    for (int nt = 0; nt < NTW; ++nt) {
                        const float* n0 = dNh + pl(k0 + L.t, col0 + 8 * nt + L.g);
                        const float* n1 = dNh + pl(k0 + 4 + L.t, col0 + 8 * nt + L.g);
                        mma3(c[nt], ah, al, __float_as_uint(n0[0]), __float_as_uint(n1[0]), __float_as_uint(n0[NP * LDN]),
                             __float_as_uint(n1[NP * LDN]));
                    }
                }
            }
            __syncthreads();           // every warp is done reading Z_l (phase c): the T planes may be overwritten
            if (busy) {
#pragma unroll
                for (int nt = 0; nt < NTW; ++nt)
#pragma unroll
                    for (int half = 0; half < 2; ++half) {
                        const int j = 16 * jt + L.g + 8 * half, col = col0 + 8 * nt + 2 * L.t;
                        const float2 v = make_float2(c[nt][2 * half], c[nt][2 * half + 1]);
                        float2 hi, lo;
                        split_f(v.x, hi.x, lo.x);
                        split_f(v.y, hi.y, lo.y);
                        *reinterpret_cast<float2*>(Th + pl(j, col)) = hi;
                        *reinterpret_cast<float2*>(Tl + pl(j, col)) = lo;
                        if (j < n) *reinterpret_cast<float2*>(dZ + hbase + (j * HD + l * GD + col)) = v;
                    }
            }
        }
        __syncthreads();
        // push dZ_l through the dense connection: dG_m[j][c'] += sum_c dZ_l[j][c] * Wn_l[128 + m*GD + c'][c]
        if (busy) {
#pragma unroll
            for (int m = 0; m < l; ++m) {
                float c[NTW][4];
#pragma unroll
                for (int nt = 0; nt < NTW; ++nt) { c[nt][0] = 0.f; c[nt][1] = 0.f; c[nt][2] = 0.f; c[nt][3] = 0.f; }
                const float* wb = wsrc + m * (GD * GD * 2) + (col0 / 8) * 128 + L.lane;
#pragma unroll 2
                for (int k0 = 0; k0 < GD; k0 += 8) {
                    uint32_t ah[4], al[4];
                    const float* pa = Th + pl(16 * jt + L.a_row, L.a_col + k0);
                    ldsm4(ah, pa);
                    ldsm4(al, pa + NP * LDN);
#pragma unroll
                    for (int nt = 0; nt < NTW; ++nt) {
                        const float* f = wb + (k0 / 8) * (GD / 8) * 128 + nt * 128;
                        mma3(c[nt], ah, al, __float_as_uint(__ldg(f)), __float_as_uint(__ldg(f + 32)),
                             __float_as_uint(__ldg(f + 64)), __float_as_uint(__ldg(f + 96)));
                    }
                }
#pragma unroll
                for (int nt = 0; nt < NTW; ++nt)
#pragma unroll
                    for (int half = 0; half < 2; ++half) {
                        float2* p = reinterpret_cast<float2*>(dGs + (TWO ? pl(16 * jt + L.g + 8 * half, m * GD + col0 + 8 * nt + 2 * L.t)
                                                                        : (16 * jt + L.g + 8 * half) * LDP + m * GD + col0 + 8 * nt + 2 * L.t));
                        float2 v = make_float2(c[nt][2 * half], c[nt][2 * half + 1]);
                        if (!first_layer) { const float2 cur = *p; v.x += cur.x; v.y += cur.y; }
                        *p = v;
                    }
            }
        }
        __syncthreads();
    }

    if (L.warp < UNITS_C) {            // dA accumulators -> shared scratch for the row-wise phase
        const int mt = L.warp / NG_C, jg = L.warp - mt * NG_C;
#pragma unroll
        for (int nt = 0; nt < NTW_C; ++nt)
#pragma unroll
            for (int half = 0; half < 2; ++half)
                *reinterpret_cast<float2*>(dAs + (16 * mt + L.g + 8 * half) * LDA + 8 * (NTW_C * jg + nt) + 2 * L.t) =
                    make_float2(cA[nt][2 * half], cA[nt][2 * half + 1]);
    }
    __syncthreads();
    // ---- attention gradient leaves the CTA: rows in groups of 8 lanes ---------------------------
#pragma unroll
    for (int r0 = 0; r0 < NP; r0 += 32) {
        const int i = r0 + L.rsub;
        if (i >= NP) continue;
        const bool rv = i < n;
        const float dr = rv ? drs[i] : 0.f;
        float p[8], dp[8];
        float dot = 0.f;
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int j = L.l8 + 8 * r;
            p[r] = 0.f; dp[r] = 0.f;
            if (r < NT8 && rv && j < n) {
                dp[r] = dAs[i * LDA + j] + dr;
                if (OUT != BK_OUT_DA) {
                    if (drop.thr_att != 0u) {     // dP = dA * keep ; P itself comes from global (the planes hold A = P * keep)
                        dp[r] *= drop_keep(drop.seed, drop.s_att, abase + i * n + j, drop.thr_att, drop.inv_att);
                        p[r] = Ab[i * n + j];
                    } else {
                        p[r] = AtS[j * LDA + i];
                    }
                    dot += dp[r] * p[r];
                }
            }
        }
        if (OUT != BK_OUT_DA) dot = group8_sum(dot);
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int j = L.l8 + 8 * r;
            if (r < NT8) {
                const float ds = (OUT == BK_OUT_DA) ? dp[r] : p[r] * (dp[r] - dot);
                if (OUT == BK_OUT_DQ) dAs[i * LDA + j] = ds;           // zeros in the padding
                else if (rv && j < n) dOut[abase + static_cast<long long>(i) * n + j] = ds;
            }
        }
    }
    if (OUT == BK_OUT_DQ) {
        // dq_h = scale (dS + dS^T) q_h   (S = scale q q^T is symmetric in q) -- one more small MMA
        constexpr int LQ = DHH + 8, Q4 = DHH / 4;
        float* Wh = dNh;               // [NP][LDA] hi / lo planes of dS + dS^T (the dN / T planes are dead)
        float* Wl = Wh + NP * LDA;
        float* qs = Wl + NP * LDA;     // [NP][LQ]  head slice of q, fp32
        for (int idx = tid; idx < NP * Q4; idx += BK_THREADS) {
            const int j = idx / Q4, k4 = (idx - j * Q4) * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (j < n) v = ld4g(q + static_cast<size_t>(node0 + j) * D + h * DHH + k4);
            *reinterpret_cast<float4*>(qs + j * LQ + k4) = v;
        }
        __syncthreads();
#pragma unroll
        for (int r0 = 0; r0 < NP; r0 += 32) {
            const int i = r0 + L.rsub;
            if (i >= NP) continue;
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                const int j = L.l8 + 8 * r;
                if (r < NT8) {
                    float hi, lo;
                    split_f(dAs[i * LDA + j] + dAs[j * LDA + i], hi, lo);
                    Wh[i * LDA + j] = hi;
                    Wl[i * LDA + j] = lo;
                }
            }
        }
        __syncthreads();
        constexpr int QT = DHH / 8;
        for (int u = L.warp; u < MT * QT; u += BK_WARPS) {
            const int mt = u / QT, nt = u - mt * QT;
            float c[4] = {0.f, 0.f, 0.f, 0.f};
            const float* pa = Wh + (16 * mt + L.a_row) * LDA + L.a_col;
            const float* qb = qs + L.t * LQ + 8 * nt + L.g;
#pragma unroll
            for (int k0 = 0; k0 < NP; k0 += 8) {
                uint32_t ah[4], al[4];
                ldsm4(ah, pa + k0);
                ldsm4(al, pa + NP * LDA + k0);
                mma3f(c, ah, al, qb[k0 * LQ], qb[(k0 + 4) * LQ]);
            }
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int i = 16 * mt + L.g + 8 * half;
                if (i < n)
                    *reinterpret_cast<float2*>(dOut + static_cast<size_t>(node0 + i) * D + h * DHH + 8 * nt + 2 * L.t) =
                        make_float2(c[2 * half] * scale, c[2 * half + 1] * scale);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
static size_t block_fwd_smem(int np, int layers, int gd) {
    const int ki = (layers - 1) * gd;
    return (2 * static_cast<size_t>(np) * (np + 4) + 2 * static_cast<size_t>(np) * (gd + 8) +
            2 * static_cast<size_t>(np) * (ki + 4) + np) * sizeof(float);
}
static size_t block_bwd_smem(int np, int layers, int gd) {
    const int ki = (layers - 1) * gd;
    size_t fl = static_cast<size_t>(np) * (np + 4) + 4 * static_cast<size_t>(np) * (gd == 64 ? gd : gd + 12) + 2 * np;
    if (layers != 2) fl += static_cast<size_t>(np) * (np + 4) + static_cast<size_t>(np) * (ki + 4);   // dA scratch, parked dG
    return fl * sizeof(float);
}

// Block kernels cover: documents of <= 64 nodes, slab 128 cut into 2 x 64 or 4 x 32 sub-layers, and -- when
// the attention is computed in-kernel -- heads of width 16 or 32.
bool block_kernels_usable(const gcgcn_batch* bt, int heads, int layers, int slab, bool mha) {
    if (slab != D || layers < 1 || slab % layers != 0) return false;
    const int gd = slab / layers;
    if (bt->max_nodes > 64 || !(gd == 32 || gd == 64)) return false;
    if (mha) {
        if (heads < 1 || D % heads != 0) return false;
        const int dh = D / heads;
        if (!(dh == 16 || dh == 32)) return false;
    }
    return true;
}

template <int GD, int DH, int MTC>
static int launch_fwd_class(const gcgcn_batch* bt, int heads, int count, int first, const int* order, const float* A,
                            const float* q, float* P, float* Z, const float* E, const float* Winner, const float* x,
                            float* G, float* F, float scale, const BlockDrop& drop, cudaStream_t st) {
    constexpr int layers = D / GD;
    const size_t smem = block_fwd_smem(16 * MTC, layers, GD);
    static std::atomic<unsigned long long> prepared{0};
    GCGCN_TRY(set_smem_once(prepared, block_fwd_kernel<GD, DH, MTC>, smem, "block_fwd"));
    block_fwd_kernel<GD, DH, MTC><<<dim3(count, heads), BK_THREADS, smem, st>>>(
        bt->node_ptr, reinterpret_cast<const long long*>(bt->pair_ptr), A, q, P, Z, E, Winner, x, G, F, heads,
        bt->total_pairs, order, first, scale, drop);
    GCGCN_CHECK_LAUNCH(DH > 0 ? "block_fwd<mha>" : "block_fwd<given>");
    return GCGCN_OK;
}

template <int GD, int DH>
static int launch_fwd_all(const gcgcn_batch* bt, int heads, const float* A, const float* q, float* P, float* Z,
                          const float* E, const float* Winner, const float* x, float* G, float* F, float scale,
                          const BlockDrop& drop, cudaStream_t st) {
    return for_each_size_class(bt, [&](int count, int first, int nmax, const int* order) -> int {
        switch ((nmax + 15) / 16) {
            case 1: return launch_fwd_class<GD, DH, 1>(bt, heads, count, first, order, A, q, P, Z, E, Winner, x, G, F, scale, drop, st);
            case 2: return launch_fwd_class<GD, DH, 2>(bt, heads, count, first, order, A, q, P, Z, E, Winner, x, G, F, scale, drop, st);
            case 3: return launch_fwd_class<GD, DH, 3>(bt, heads, count, first, order, A, q, P, Z, E, Winner, x, G, F, scale, drop, st);
            case 4: return launch_fwd_class<GD, DH, 4>(bt, heads, count, first, order, A, q, P, Z, E, Winner, x, G, F, scale, drop, st);
            default: return fail(GCGCN_ERR_UNSUPPORTED, "block_fwd: %d nodes > 64", nmax);
        }
    });
}

// A != nullptr: attention given (q, P unused).  A == nullptr: MHA from q, P written.
static int launch_winner_frag(const float* Winner, int heads, int layers, float* frag_ws, cudaStream_t st) {
    if (layers < 2) return GCGCN_OK;
    if (frag_ws == nullptr) return fail(GCGCN_ERR_WORKSPACE, "block kernels: no workspace for the fragment-ordered weights");
    const size_t half = block_frag_floats(heads, layers) / 2;
    winner_frag_kernel<<<dim3(heads * layers, 8), 256, 0, st>>>(Winner, layers, D / layers, frag_ws, frag_ws + half);
    GCGCN_CHECK_LAUNCH("winner_frag");
    return GCGCN_OK;
}

// gcn_tile.cu: the same block on packed 128-row tcgen05 tiles (MHA attention, two sub-layers, head width 16, eval mode)
bool tile_blocks_enabled();
size_t tile_wblob_bytes(int heads);
int launch_tile_fwd(const gcgcn_batch* bt, int heads, int layers, const float* q, float* P, float* Z, const float* E,
                    const float* Winner_rowmajor, const float* x, float* G, float* F, void* wblob_ws, cudaStream_t st);

int launch_block_fwd(const gcgcn_batch* bt, int heads, int layers, const float* A, const float* q, float* P,
                     float* Z, const float* E, const float* Winner_rowmajor, const float* x, float* G, float* F,
                     float* frag_ws, const BlockDrop& drop, cudaStream_t st) {
    if (bt->num_docs == 0) return GCGCN_OK;
    if (A == nullptr && layers == 2 && (heads == 8 || heads == 4) && drop.thr_att == 0u && drop.thr_gcn == 0u && bt->tile_doc != nullptr &&
        bt->num_tiles > 0 && bt->row_doc != nullptr && frag_ws != nullptr &&
        tile_wblob_bytes(heads) <= block_frag_floats(heads, layers) * sizeof(float) && tile_blocks_enabled())
        return launch_tile_fwd(bt, heads, layers, q, P, Z, E, Winner_rowmajor, x, G, F, frag_ws, st);
    GCGCN_TRY(launch_winner_frag(Winner_rowmajor, heads, layers, frag_ws, st));
    const float* Winner = frag_ws;                      // forward-ordered half
    const int gd = D / layers;
    const int dh = A != nullptr ? 0 : D / heads;
    const float scale = dh > 0 ? 1.0f / sqrtf(static_cast<float>(dh)) : 1.f;
#define GCGCN_BK_FWD(GD_, DH_) \
    if (gd == GD_ && dh == DH_) return launch_fwd_all<GD_, DH_>(bt, heads, A, q, P, Z, E, Winner, x, G, F, scale, drop, st);
    GCGCN_BK_FWD(64, 0)
    GCGCN_BK_FWD(64, 16)
    GCGCN_BK_FWD(64, 32)
    GCGCN_BK_FWD(32, 0)
    GCGCN_BK_FWD(32, 16)
    GCGCN_BK_FWD(32, 32)
#undef GCGCN_BK_FWD
    return fail(GCGCN_ERR_UNSUPPORTED, "block_fwd: sub-layer width %d / head width %d not supported", gd, dh);
}

template <int GD, int DH, int OUT, int MTC>
static int launch_bwd_class(const gcgcn_batch* bt, int heads, int count, int first, const int* order, const float* A,
                            const float* q, const float* Z, const float* G, const float* Winner, const float* dF,
                            float* dZ, float* dE, float* dOut, float scale, const BlockDrop& drop, cudaStream_t st) {
    constexpr int layers = D / GD;
    const size_t smem = block_bwd_smem(16 * MTC, layers, GD);
    static std::atomic<unsigned long long> prepared{0};
    GCGCN_TRY(set_smem_once(prepared, block_bwd_kernel<GD, DH, OUT, MTC>, smem, "block_bwd"));
    block_bwd_kernel<GD, DH, OUT, MTC><<<dim3(count, heads), BK_THREADS, smem, st>>>(
        bt->node_ptr, reinterpret_cast<const long long*>(bt->pair_ptr), A, q, Z, G, Winner, dF, dZ, dE, dOut, heads,
        bt->total_pairs, order, first, scale, drop);
    GCGCN_CHECK_LAUNCH(OUT == BK_OUT_DQ ? "block_bwd<dq>" : (OUT == BK_OUT_DS ? "block_bwd<dS>" : "block_bwd<dA>"));
    return GCGCN_OK;
}

template <int GD, int DH, int OUT>
static int launch_bwd_all(const gcgcn_batch* bt, int heads, const float* A, const float* q, const float* Z,
                          const float* G, const float* Winner, const float* dF, float* dZ, float* dE, float* dOut,
                          float scale, const BlockDrop& drop, cudaStream_t st) {
    return for_each_size_class(bt, [&](int count, int first, int nmax, const int* order) -> int {
        switch ((nmax + 15) / 16) {
            case 1: return launch_bwd_class<GD, DH, OUT, 1>(bt, heads, count, first, order, A, q, Z, G, Winner, dF, dZ, dE, dOut, scale, drop, st);
            case 2: return launch_bwd_class<GD, DH, OUT, 2>(bt, heads, count, first, order, A, q, Z, G, Winner, dF, dZ, dE, dOut, scale, drop, st);
            case 3: return launch_bwd_class<GD, DH, OUT, 3>(bt, heads, count, first, order, A, q, Z, G, Winner, dF, dZ, dE, dOut, scale, drop, st);
            case 4: return launch_bwd_class<GD, DH, OUT, 4>(bt, heads, count, first, order, A, q, Z, G, Winner, dF, dZ, dE, dOut, scale, drop, st);
            default: return fail(GCGCN_ERR_UNSUPPORTED, "block_bwd: %d nodes > 64", nmax);
        }
    });
}

// out_mode: BK_OUT_DA -> dOut = dA [heads][total_pairs]; BK_OUT_DS -> dOut = dS (same shape; A must be a softmax
// output); BK_OUT_DQ -> dOut = dq [total_nodes][128] (A = the MHA probabilities, q their query projection).
int launch_block_bwd(const gcgcn_batch* bt, int heads, int layers, int out_mode, const float* A, const float* q,
                     const float* Z, const float* G, const float* Winner_rowmajor, const float* dF, float* dZ, float* dE,
                     float* dOut, float* frag_ws, const BlockDrop& drop, cudaStream_t st) {
    if (bt->num_docs == 0) return GCGCN_OK;
    GCGCN_TRY(launch_winner_frag(Winner_rowmajor, heads, layers, frag_ws, st));
    const float* Winner = frag_ws == nullptr ? nullptr : frag_ws + block_frag_floats(heads, layers) / 2;   // backward-ordered half
    const int gd = D / layers;
    const int dh = out_mode == BK_OUT_DQ ? D / heads : 0;
    const float scale = dh > 0 ? 1.0f / sqrtf(static_cast<float>(dh)) : 1.f;
#define GCGCN_BK_BWD(GD_, DH_, OUT_)                      \
    if (gd == GD_ && dh == DH_ && out_mode == OUT_)       \
        return launch_bwd_all<GD_, DH_, OUT_>(bt, heads, A, q, Z, G, Winner, dF, dZ, dE, dOut, scale, drop, st);
    GCGCN_BK_BWD(64, 0, BK_OUT_DA)
    GCGCN_BK_BWD(32, 0, BK_OUT_DA)
    GCGCN_BK_BWD(64, 0, BK_OUT_DS)
    GCGCN_BK_BWD(32, 0, BK_OUT_DS)
    GCGCN_BK_BWD(64, 16, BK_OUT_DQ)
    GCGCN_BK_BWD(64, 32, BK_OUT_DQ)
    GCGCN_BK_BWD(32, 16, BK_OUT_DQ)
    GCGCN_BK_BWD(32, 32, BK_OUT_DQ)
#undef GCGCN_BK_BWD
    return fail(GCGCN_ERR_UNSUPPORTED, "block_bwd: sub-layer width %d / head width %d / mode %d not supported", gd, dh,
                out_mode);
}

}  // namespace gcgcn
