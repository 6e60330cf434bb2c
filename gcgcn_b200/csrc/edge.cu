// Edge pass ("K_edge_reduce") and the attention-row kernels that hang off it.
//
// The n x n x 128 edge tensor of a document is the only operand of the hot path whose bytes
// matter (SURVEY.md section 8d).  Everything the reference does with it collapses to two
// reductions along the feature / column axis:
//   s_ij  = v . e_ij            (GATAttention's linear_edge_r + wt, G:161-162, collapsed)
//   ebar_i = mean_j e_ij        (GraphConv's einsum + mean, G:40-41, collapsed)
// so one streaming pass per direction is all the HBM traffic the path needs: forward reads e
// once; backward re-reads e0 once (for dv) and writes de once.  One CTA owns one (doc, i) row:
// its n vectors of 128 features are read with 128-bit loads, a warp per vector.
#include "common.cuh"

namespace gcgcn {

constexpr int EDGE_THREADS = 128;
constexpr int EDGE_WARPS = EDGE_THREADS / WARP;
constexpr int EDGE_UNROLL = 4;

struct RowInfo {
    int n;            // entities of the document
    int i;            // row inside the document
    int node0;        // first node row of the document
    long long prow;   // pair index of (i, 0)
};

__device__ __forceinline__ RowInfo row_info(int r, const int* __restrict__ node_ptr,
                                            const long long* __restrict__ pair_ptr,
                                            const int* __restrict__ row_doc) {
    RowInfo ri;
    int b = row_doc[r];
    ri.node0 = node_ptr[b];
    ri.n = node_ptr[b + 1] - ri.node0;
    ri.i = r - ri.node0;
    ri.prow = pair_ptr[b] + static_cast<long long>(ri.i) * ri.n;
    return ri;
}

// ---------------------------------------------------------------------------------------------
// ux[r] = x[r,:] . u + c        (node half of the GAT energy, G:159-160 + G:162 collapsed)
__global__ void __launch_bounds__(256) node_score_kernel(const float* __restrict__ x,
                                                          const float* __restrict__ u,
                                                          const float* __restrict__ c,
                                                          float* __restrict__ ux, int rows) {
    int lane = threadIdx.x & 31;
    int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int nwarps = (gridDim.x * blockDim.x) >> 5;
    float4 u4 = *reinterpret_cast<const float4*>(u + lane * 4);
    float c0 = c ? *c : 0.f;
    for (int r = warp; r < rows; r += nwarps) {
        float4 a = *reinterpret_cast<const float4*>(x + static_cast<size_t>(r) * D + lane * 4);
        float p = a.x * u4.x + a.y * u4.y + a.z * u4.z + a.w * u4.w;
        p = warp_sum(p);
        if (lane == 0) ux[r] = p + c0;
    }
}

// ---------------------------------------------------------------------------------------------
// forward edge pass: one CTA per (doc, i) row
template <typename T, bool WITH_SCORE>
__global__ void __launch_bounds__(EDGE_THREADS)
edge_row_fwd_kernel(const T* __restrict__ e, const int* __restrict__ node_ptr,
                    const long long* __restrict__ pair_ptr, const int* __restrict__ row_doc,
                    const float* __restrict__ v, const float* __restrict__ ux,
                    const uint8_t* __restrict__ mask, const float* __restrict__ keep,
                    float* __restrict__ P, float* __restrict__ A, float* __restrict__ ebar) {
    extern __shared__ float smem[];
    float* part = smem;                     // [EDGE_WARPS][D] partial column sums
    float* s = smem + EDGE_WARPS * D;       // [n] energies
    __shared__ float red[EDGE_WARPS];

    const int r = blockIdx.x;
    const RowInfo ri = row_info(r, node_ptr, pair_ptr, row_doc);
    const int n = ri.n;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const T* erow = e + ri.prow * D + lane * 4;

    float4 v4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (WITH_SCORE) v4 = *reinterpret_cast<const float4*>(v + lane * 4);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);

    for (int jb = warp; jb < n; jb += EDGE_WARPS * EDGE_UNROLL) {
        float4 t[EDGE_UNROLL];
#pragma unroll
        for (int k = 0; k < EDGE_UNROLL; ++k) {
            int j = jb + k * EDGE_WARPS;
            t[k] = (j < n) ? Vec4<T>::load(erow + static_cast<size_t>(j) * D)
                           : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int k = 0; k < EDGE_UNROLL; ++k) {
            int j = jb + k * EDGE_WARPS;
            acc.x += t[k].x; acc.y += t[k].y; acc.z += t[k].z; acc.w += t[k].w;
            if (WITH_SCORE) {
                float p = t[k].x * v4.x + t[k].y * v4.y + t[k].z * v4.z + t[k].w * v4.w;
                p = warp_sum(p);
                if (lane == 0 && j < n) s[j] = p;
            }
        }
    }
    *reinterpret_cast<float4*>(part + warp * D + lane * 4) = acc;
    __syncthreads();
    {
        int t = threadIdx.x;  // EDGE_THREADS == D
        float sum = 0.f;
#pragma unroll
        for (int w = 0; w < EDGE_WARPS; ++w) sum += part[w * D + t];
        ebar[static_cast<size_t>(r) * D + t] = sum / static_cast<float>(n);
    }
    if (!WITH_SCORE) return;

    // energy_ij = s_ij + ux_j  -> row softmax over all n columns (G:165).  The reference never
    // applies its mask (G:163-164); `mask` is non-null only when the caller opted in.
    float m = -INFINITY;
    for (int j = threadIdx.x; j < n; j += EDGE_THREADS) {
        float en = s[j] + ux[ri.node0 + j];
        if (mask != nullptr && mask[ri.prow + j]) en = -100000.0f;
        s[j] = en;
        m = fmaxf(m, en);
    }
    m = warp_max(m);
    if (lane == 0) red[warp] = m;
    __syncthreads();
    m = red[0];
#pragma unroll
    for (int w = 1; w < EDGE_WARPS; ++w) m = fmaxf(m, red[w]);
    __syncthreads();
    float z = 0.f;
    for (int j = threadIdx.x; j < n; j += EDGE_THREADS) {
        float ex = expf(s[j] - m);
        s[j] = ex;
        z += ex;
    }
    z = warp_sum(z);
    if (lane == 0) red[warp] = z;
    __syncthreads();
    z = 0.f;
#pragma unroll
    for (int w = 0; w < EDGE_WARPS; ++w) z += red[w];
    for (int j = threadIdx.x; j < n; j += EDGE_THREADS) {
        float p = s[j] / z;
        P[ri.prow + j] = p;
        if (keep != nullptr) A[ri.prow + j] = p * keep[ri.prow + j];
        else if (A != P) A[ri.prow + j] = p;
    }
}

// ---------------------------------------------------------------------------------------------
// backward edge pass, persistent: de_ij = dS_ij * v + debar_i / n ; dv += sum_ij dS_ij e_ij
template <typename T, bool WITH_SCORE>
__global__ void __launch_bounds__(EDGE_THREADS)
edge_row_bwd_kernel(const T* __restrict__ e, const int* __restrict__ node_ptr,
                    const long long* __restrict__ pair_ptr, const int* __restrict__ row_doc,
                    const float* __restrict__ v, const float* __restrict__ dS,
                    const float* __restrict__ debar, T* __restrict__ de,
                    float* __restrict__ dv_partial, int total_nodes) {
    __shared__ float part[EDGE_WARPS * D];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float4 v4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (WITH_SCORE) v4 = *reinterpret_cast<const float4*>(v + lane * 4);
    float4 dv = make_float4(0.f, 0.f, 0.f, 0.f);

    for (int r = blockIdx.x; r < total_nodes; r += gridDim.x) {
        const RowInfo ri = row_info(r, node_ptr, pair_ptr, row_doc);
        const int n = ri.n;
        float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
        if (debar != nullptr) {
            g = *reinterpret_cast<const float4*>(debar + static_cast<size_t>(r) * D + lane * 4);
            float inv = 1.0f / static_cast<float>(n);
            g.x *= inv; g.y *= inv; g.z *= inv; g.w *= inv;
        }
        const size_t base = static_cast<size_t>(ri.prow) * D + lane * 4;
        for (int jb = warp; jb < n; jb += EDGE_WARPS * EDGE_UNROLL) {
            float4 t[EDGE_UNROLL];
            float ds[EDGE_UNROLL];
#pragma unroll
            for (int k = 0; k < EDGE_UNROLL; ++k) {
                int j = jb + k * EDGE_WARPS;
                if (WITH_SCORE && j < n) {
                    t[k] = Vec4<T>::load(e + base + static_cast<size_t>(j) * D);
                    ds[k] = dS[ri.prow + j];
                } else {
                    t[k] = make_float4(0.f, 0.f, 0.f, 0.f);
                    ds[k] = 0.f;
                }
            }
#pragma unroll
            for (int k = 0; k < EDGE_UNROLL; ++k) {
                int j = jb + k * EDGE_WARPS;
                if (j < n) {
                    float4 o = g;
                    if (WITH_SCORE) {
                        o.x += ds[k] * v4.x; o.y += ds[k] * v4.y; o.z += ds[k] * v4.z; o.w += ds[k] * v4.w;
                        dv.x += ds[k] * t[k].x; dv.y += ds[k] * t[k].y;
                        dv.z += ds[k] * t[k].z; dv.w += ds[k] * t[k].w;
                    }
                    Vec4<T>::store(de + base + static_cast<size_t>(j) * D, o);
                }
            }
        }
    }
    if (!WITH_SCORE) return;
    *reinterpret_cast<float4*>(part + warp * D + lane * 4) = dv;
    __syncthreads();
    int t = threadIdx.x;
    float sum = 0.f;
#pragma unroll
    for (int w = 0; w < EDGE_WARPS; ++w) sum += part[w * D + t];
    dv_partial[static_cast<size_t>(blockIdx.x) * D + t] = sum;
}

// ---------------------------------------------------------------------------------------------
// softmax backward over attention rows, one warp per (head, node row):
//   dP = dA * keep ; dS = P * (dP - sum_j dP_j P_j)   (masked entries carry no gradient)
__global__ void __launch_bounds__(256)
softmax_bwd_kernel(const int* __restrict__ node_ptr, const long long* __restrict__ pair_ptr,
                   const int* __restrict__ row_doc, const float* __restrict__ P,
                   const float* __restrict__ keep, const float* __restrict__ dA,
                   const uint8_t* __restrict__ mask, float* __restrict__ dS, int total_nodes,
                   long long total_pairs, int heads) {
    const int lane = threadIdx.x & 31;
    const long long gw = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const long long nw = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
    const long long rows = static_cast<long long>(total_nodes) * heads;
    for (long long w = gw; w < rows; w += nw) {
        const int h = static_cast<int>(w / total_nodes);
        const int r = static_cast<int>(w - static_cast<long long>(h) * total_nodes);
        const RowInfo ri = row_info(r, node_ptr, pair_ptr, row_doc);
        const long long off = static_cast<long long>(h) * total_pairs + ri.prow;
        if ((ri.n & 3) == 0 && (off & 3) == 0 && mask == nullptr) {      // 16-byte accesses: rows of 4 k floats
            float dot = 0.f;
            for (int j = lane * 4; j < ri.n; j += 4 * WARP) {
                float4 dp = *reinterpret_cast<const float4*>(dA + off + j);
                if (keep != nullptr) {
                    const float4 k4 = *reinterpret_cast<const float4*>(keep + off + j);
                    dp.x *= k4.x; dp.y *= k4.y; dp.z *= k4.z; dp.w *= k4.w;
                }
                const float4 p4 = *reinterpret_cast<const float4*>(P + off + j);
                dot += dp.x * p4.x + dp.y * p4.y + dp.z * p4.z + dp.w * p4.w;
            }
            dot = warp_sum(dot);
            for (int j = lane * 4; j < ri.n; j += 4 * WARP) {
                float4 dp = *reinterpret_cast<const float4*>(dA + off + j);
                if (keep != nullptr) {
                    const float4 k4 = *reinterpret_cast<const float4*>(keep + off + j);
                    dp.x *= k4.x; dp.y *= k4.y; dp.z *= k4.z; dp.w *= k4.w;
                }
                const float4 p4 = *reinterpret_cast<const float4*>(P + off + j);
                *reinterpret_cast<float4*>(dS + off + j) = make_float4(p4.x * (dp.x - dot), p4.y * (dp.y - dot),
                                                                       p4.z * (dp.z - dot), p4.w * (dp.w - dot));
            }
            continue;
        }
        float dot = 0.f;
        for (int j = lane; j < ri.n; j += WARP) {
            float dp = dA[off + j];
            if (keep != nullptr) dp *= keep[off + j];
            dot += dp * P[off + j];
        }
        dot = warp_sum(dot);
        for (int j = lane; j < ri.n; j += WARP) {
            float dp = dA[off + j];
            if (keep != nullptr) dp *= keep[off + j];
            float ds = P[off + j] * (dp - dot);
            if (mask != nullptr && mask[ri.prow + j]) ds = 0.f;
            dS[off + j] = ds;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// node half of the GAT backward: dux_j = sum_i dS_ij ; dx_j = dux_j * u ; du += dux_j x_j ; dc += dux_j
// one warp per node row, persistent; partial[blockIdx][D + 1] holds (du, dc) per CTA.
constexpr int NODE_BWD_THREADS = 256;
__global__ void __launch_bounds__(NODE_BWD_THREADS)
gat_node_bwd_kernel(const int* __restrict__ node_ptr, const long long* __restrict__ pair_ptr,
                    const int* __restrict__ row_doc, const float* __restrict__ dS,
                    const float* __restrict__ x, const float* __restrict__ u,
                    float* __restrict__ dx, float* __restrict__ partial, int total_nodes) {
    constexpr int NW = NODE_BWD_THREADS / WARP;
    __shared__ float part[NW * (D + 1)];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float4 u4 = *reinterpret_cast<const float4*>(u + lane * 4);
    float4 du = make_float4(0.f, 0.f, 0.f, 0.f);
    float dc = 0.f;
    for (int r = blockIdx.x * NW + warp; r < total_nodes; r += gridDim.x * NW) {
        const int b = row_doc[r];
        const int node0 = node_ptr[b];
        const int n = node_ptr[b + 1] - node0;
        const int j = r - node0;
        const float* col = dS + pair_ptr[b] + j;
        float sum = 0.f;
        for (int i = lane; i < n; i += WARP) sum += col[static_cast<size_t>(i) * n];
        sum = warp_sum(sum);
        float4 xv = *reinterpret_cast<const float4*>(x + static_cast<size_t>(r) * D + lane * 4);
        float4 o = make_float4(sum * u4.x, sum * u4.y, sum * u4.z, sum * u4.w);
        *reinterpret_cast<float4*>(dx + static_cast<size_t>(r) * D + lane * 4) = o;
        du.x += sum * xv.x; du.y += sum * xv.y; du.z += sum * xv.z; du.w += sum * xv.w;
        dc += sum;
    }
    float* mine = part + warp * (D + 1);
    mine[lane * 4 + 0] = du.x; mine[lane * 4 + 1] = du.y;
    mine[lane * 4 + 2] = du.z; mine[lane * 4 + 3] = du.w;
    if (lane == 0) mine[D] = dc;
    __syncthreads();
    for (int t = threadIdx.x; t < D + 1; t += NODE_BWD_THREADS) {
        float sum = 0.f;
#pragma unroll
        for (int w = 0; w < NW; ++w) sum += part[w * (D + 1) + t];
        partial[static_cast<size_t>(blockIdx.x) * (D + 1) + t] = sum;
    }
}

// out[c] = sum_p partial[p][c]  (deterministic second stage of every cross-CTA reduction)
__global__ void __launch_bounds__(1024)
reduce_partials_kernel(const float* __restrict__ partial, int parts, int width,
                       float* __restrict__ out0, int width0, float* __restrict__ out1) {
    // block = 32 columns x 32 row lanes; lane r adds parts r, r+32, ... in order on eight interleaved chains (eight
    // loads in flight: with two, the 2368 partials of the edge pass were 37 dependent round trips, 15 us), then the
    // chains and the 32 lane sums are added in a fixed order: the result does not depend on scheduling
    __shared__ float red[32][33];
    const int cl = threadIdx.x & 31, rl = threadIdx.x >> 5;
    const int c = blockIdx.x * 32 + cl;
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (c < width) {
        int p = rl;
        for (; p + 7 * 32 < parts; p += 8 * 32) {
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] += partial[static_cast<size_t>(p + 32 * i) * width + c];
        }
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if (p + 32 * i < parts) acc[i] += partial[static_cast<size_t>(p + 32 * i) * width + c];
    }
    const float s0 = (acc[0] + acc[1]) + (acc[2] + acc[3]), s1 = (acc[4] + acc[5]) + (acc[6] + acc[7]);
    red[rl][cl] = s0 + s1;
    __syncthreads();
    if (rl == 0 && c < width) {
        float t = 0.f;
#pragma unroll
        for (int r = 0; r < 32; ++r) t += red[r][cl];
        if (c < width0) out0[c] = t;
        else if (out1 != nullptr) out1[c - width0] = t;
    }
}

// ---------------------------------------------------------------------------------------------
// host launchers
int launch_node_score(const float* x, const float* u, const float* c, float* ux, int rows,
                      cudaStream_t st) {
    if (rows == 0) return GCGCN_OK;
    int blocks = min(ceil_div(rows, 8), sm_count() * 8);
    node_score_kernel<<<blocks, 256, 0, st>>>(x, u, c, ux, rows);
    GCGCN_CHECK_LAUNCH("node_score");
    return GCGCN_OK;
}

template <typename T>
static int edge_fwd_t(const gcgcn_batch* bt, const T* e, const float* v, const float* ux,
                      const uint8_t* mask, const float* keep, float* P, float* A, float* ebar,
                      cudaStream_t st) {
    size_t smem = (EDGE_WARPS * D + bt->max_nodes) * sizeof(float);
    if (v != nullptr) {
        GCGCN_TRY(set_smem(edge_row_fwd_kernel<T, true>, smem, "edge_fwd smem"));
        edge_row_fwd_kernel<T, true><<<bt->total_nodes, EDGE_THREADS, smem, st>>>(
            e, bt->node_ptr, reinterpret_cast<const long long*>(bt->pair_ptr), bt->row_doc, v, ux,
            mask, keep, P, A, ebar);
        GCGCN_CHECK_LAUNCH("edge_row_fwd<score+mean>");
    } else {
        edge_row_fwd_kernel<T, false><<<bt->total_nodes, EDGE_THREADS, EDGE_WARPS * D * sizeof(float), st>>>(
            e, bt->node_ptr, reinterpret_cast<const long long*>(bt->pair_ptr), bt->row_doc, nullptr,
            nullptr, nullptr, nullptr, nullptr, nullptr, ebar);
        GCGCN_CHECK_LAUNCH("edge_row_fwd<mean>");
    }
    return GCGCN_OK;
}

int launch_edge_fwd(const gcgcn_batch* bt, const void* e, int dtype, const float* v, const float* ux,
                    const uint8_t* mask, const float* keep, float* P, float* A, float* ebar,
                    cudaStream_t st) {
    if (bt->total_nodes == 0) return GCGCN_OK;
    if (dtype == GCGCN_F32)
        return edge_fwd_t<float>(bt, static_cast<const float*>(e), v, ux, mask, keep, P, A, ebar, st);
    if (dtype == GCGCN_BF16)
        return edge_fwd_t<__nv_bfloat16>(bt, static_cast<const __nv_bfloat16*>(e), v, ux, mask, keep,
                                         P, A, ebar, st);
    return fail(GCGCN_ERR_UNSUPPORTED, "edge dtype %d not supported", dtype);
}

int edge_bwd_grid() { return sm_count() * 16; }

template <typename T>
static int edge_bwd_t(const gcgcn_batch* bt, const T* e, const float* v, const float* dS,
                      const float* debar, T* de, float* dv_partial, cudaStream_t st) {
    int grid = min(edge_bwd_grid(), bt->total_nodes);
    const long long* pp = reinterpret_cast<const long long*>(bt->pair_ptr);
    if (dS != nullptr) {
        edge_row_bwd_kernel<T, true><<<grid, EDGE_THREADS, 0, st>>>(e, bt->node_ptr, pp, bt->row_doc, v,
                                                                    dS, debar, de, dv_partial,
                                                                    bt->total_nodes);
        GCGCN_CHECK_LAUNCH("edge_row_bwd<score+mean>");
    } else {
        edge_row_bwd_kernel<T, false><<<grid, EDGE_THREADS, 0, st>>>(nullptr, bt->node_ptr, pp,
                                                                     bt->row_doc, nullptr, nullptr,
                                                                     debar, de, nullptr,
                                                                     bt->total_nodes);
        GCGCN_CHECK_LAUNCH("edge_row_bwd<mean>");
    }
    return GCGCN_OK;
}

// dv_partial: [min(edge_bwd_grid(), total_nodes)][D] when dS != nullptr
int launch_edge_bwd(const gcgcn_batch* bt, const void* e, int dtype, const float* v, const float* dS,
                    const float* debar, void* de, float* dv_partial, cudaStream_t st) {
    if (bt->total_nodes == 0) return GCGCN_OK;
    if (dtype == GCGCN_F32)
        return edge_bwd_t<float>(bt, static_cast<const float*>(e), v, dS, debar,
                                 static_cast<float*>(de), dv_partial, st);
    if (dtype == GCGCN_BF16)
        return edge_bwd_t<__nv_bfloat16>(bt, static_cast<const __nv_bfloat16*>(e), v, dS, debar,
                                         static_cast<__nv_bfloat16*>(de), dv_partial, st);
    return fail(GCGCN_ERR_UNSUPPORTED, "edge dtype %d not supported", dtype);
}

int launch_softmax_bwd(const gcgcn_batch* bt, int heads, const float* P, const float* keep,
                       const float* dA, const uint8_t* mask, float* dS, cudaStream_t st) {
    long long rows = static_cast<long long>(bt->total_nodes) * heads;
    if (rows == 0) return GCGCN_OK;
    int blocks = static_cast<int>(std::min<long long>((rows + 7) / 8, static_cast<long long>(sm_count()) * 16));
    softmax_bwd_kernel<<<blocks, 256, 0, st>>>(bt->node_ptr,
                                               reinterpret_cast<const long long*>(bt->pair_ptr),
                                               bt->row_doc, P, keep, dA, mask, dS, bt->total_nodes,
                                               bt->total_pairs, heads);
    GCGCN_CHECK_LAUNCH("softmax_bwd");
    return GCGCN_OK;
}

int node_bwd_grid() { return sm_count() * 4; }

// partial: [node_bwd_grid()][D+1]
int launch_gat_node_bwd(const gcgcn_batch* bt, const float* dS, const float* x, const float* u,
                        float* dx, float* partial, int* parts_out, cudaStream_t st) {
    int grid = min(node_bwd_grid(), max(1, ceil_div(bt->total_nodes, NODE_BWD_THREADS / WARP)));
    *parts_out = grid;
    gat_node_bwd_kernel<<<grid, NODE_BWD_THREADS, 0, st>>>(
        bt->node_ptr, reinterpret_cast<const long long*>(bt->pair_ptr), bt->row_doc, dS, x, u, dx,
        partial, bt->total_nodes);
    GCGCN_CHECK_LAUNCH("gat_node_bwd");
    return GCGCN_OK;
}

int launch_reduce_partials(const float* partial, int parts, int width, float* out0, int width0,
                           float* out1, cudaStream_t st) {
    reduce_partials_kernel<<<ceil_div(width, 32), 1024, 0, st>>>(partial, parts, width, out0, width0,
                                                                out1);
    GCGCN_CHECK_LAUNCH("reduce_partials");
    return GCGCN_OK;
}

}  // namespace gcgcn
