// MultiHeadAttention score kernels (G:133-142): per (document, head) CTA.
//   P_h = softmax_j( q_h[i] . q_h[j] / sqrt(d_h) )      -- the key is the query projection (G:137)
//   A_h = P_h * keep_h
// The q projection itself (x Wq^T + bq over every node row of the batch) is a dense GEMM and is
// done by the caller; these kernels only touch the n x d_h head slice and the n x n map.
#include "common.cuh"

namespace gcgcn {

constexpr int MHA_THREADS = 256;
constexpr int MHA_WARPS = MHA_THREADS / WARP;

// smem: qs [n][dh+1] (padded: lanes walk rows), rowbuf [MHA_WARPS][n]
template <int DH>
__global__ void __launch_bounds__(MHA_THREADS)
mha_fwd_kernel(const int* __restrict__ node_ptr, const long long* __restrict__ pair_ptr,
               const float* __restrict__ q, const float* __restrict__ keep, float* __restrict__ P,
               float* __restrict__ A, long long total_pairs, float scale) {
    extern __shared__ float smem[];
    const int b = blockIdx.x, h = blockIdx.y;
    const int node0 = node_ptr[b];
    const int n = node_ptr[b + 1] - node0;
    constexpr int LD = DH + 1;
    float* qs = smem;
    float* rowbuf = smem + static_cast<size_t>(n) * LD;
    for (int t = threadIdx.x; t < n * DH; t += MHA_THREADS) {
        int j = t / DH, k = t - j * DH;
        qs[j * LD + k] = q[static_cast<size_t>(node0 + j) * D + h * DH + k];
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* buf = rowbuf + static_cast<size_t>(warp) * n;
    const long long base = static_cast<long long>(h) * total_pairs + pair_ptr[b];
    for (int i = warp; i < n; i += MHA_WARPS) {
        float qi[DH];
#pragma unroll
        for (int k = 0; k < DH; ++k) qi[k] = qs[i * LD + k];
        float m = -INFINITY;
        for (int j = lane; j < n; j += WARP) {
            float s = 0.f;
#pragma unroll
            for (int k = 0; k < DH; ++k) s += qi[k] * qs[j * LD + k];
            s *= scale;
            buf[j] = s;
            m = fmaxf(m, s);
        }
        m = warp_max(m);
        float z = 0.f;
        for (int j = lane; j < n; j += WARP) {
            float ex = expf(buf[j] - m);
            buf[j] = ex;
            z += ex;
        }
        z = warp_sum(z);
        const long long off = base + static_cast<long long>(i) * n;
        for (int j = lane; j < n; j += WARP) {
            float p = buf[j] / z;
            P[off + j] = p;
            if (keep != nullptr) A[off + j] = p * keep[off + j];
            else if (A != P) A[off + j] = p;
        }
        __syncwarp();
    }
}

// dq_h[i,:] = scale * sum_j (dS_ij + dS_ji) q_h[j,:]       (S = scale * q q^T is symmetric in q)
template <int DH>
__global__ void __launch_bounds__(MHA_THREADS)
mha_bwd_kernel(const int* __restrict__ node_ptr, const long long* __restrict__ pair_ptr,
               const float* __restrict__ q, const float* __restrict__ dS, float* __restrict__ dq,
               long long total_pairs, float scale) {
    extern __shared__ float smem[];
    const int b = blockIdx.x, h = blockIdx.y;
    const int node0 = node_ptr[b];
    const int n = node_ptr[b + 1] - node0;
    constexpr int LD = DH + 1;
    float* qs = smem;
    float* rowbuf = smem + static_cast<size_t>(n) * LD;
    for (int t = threadIdx.x; t < n * DH; t += MHA_THREADS) {
        int j = t / DH, k = t - j * DH;
        qs[j * LD + k] = q[static_cast<size_t>(node0 + j) * D + h * DH + k];
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* buf = rowbuf + static_cast<size_t>(warp) * n;
    const float* g = dS + static_cast<long long>(h) * total_pairs + pair_ptr[b];
    constexpr int GROUPS = WARP / DH;  // DH = 16 -> 2 half-warps walk alternate j; DH = 32 -> 1
    const int k = lane % DH, grp = lane / DH;
    for (int i = warp; i < n; i += MHA_WARPS) {
        for (int j = lane; j < n; j += WARP)
            buf[j] = g[static_cast<size_t>(i) * n + j] + g[static_cast<size_t>(j) * n + i];
        __syncwarp();
        float acc = 0.f;
        for (int j = grp; j < n; j += GROUPS) acc += buf[j] * qs[j * LD + k];
        if (GROUPS == 2) acc += __shfl_xor_sync(0xffffffffu, acc, 16);
        if (GROUPS == 4) {
            acc += __shfl_xor_sync(0xffffffffu, acc, 16);
            acc += __shfl_xor_sync(0xffffffffu, acc, 8);
        }
        if (grp == 0) dq[static_cast<size_t>(node0 + i) * D + h * DH + k] = acc * scale;
        __syncwarp();
    }
}

static size_t mha_smem(int n, int dh) {
    return (static_cast<size_t>(n) * (dh + 1) + static_cast<size_t>(MHA_WARPS) * n) * sizeof(float);
}

int launch_mha_fwd(const gcgcn_batch* bt, int heads, const float* q, const float* keep, float* P,
                   float* A, cudaStream_t st) {
    if (bt->num_docs == 0) return GCGCN_OK;
    const int dh = D / heads;
    const float scale = 1.0f / sqrtf(static_cast<float>(dh));
    const size_t smem = mha_smem(bt->max_nodes, dh);
    dim3 grid(bt->num_docs, heads);
    const long long* pp = reinterpret_cast<const long long*>(bt->pair_ptr);
#define GCGCN_MHA_FWD(DH)                                                                         \
    case DH:                                                                                      \
        GCGCN_TRY(set_smem(mha_fwd_kernel<DH>, smem, "mha_fwd"));                                 \
        mha_fwd_kernel<DH><<<grid, MHA_THREADS, smem, st>>>(bt->node_ptr, pp, q, keep, P, A,      \
                                                            bt->total_pairs, scale);              \
        break;
    switch (dh) {
        GCGCN_MHA_FWD(8)
        GCGCN_MHA_FWD(16)
        GCGCN_MHA_FWD(32)
        default:
            return fail(GCGCN_ERR_UNSUPPORTED, "head_num %d (d_h = %d) not supported; use 4, 8 or 16",
                        heads, dh);
    }
#undef GCGCN_MHA_FWD
    GCGCN_CHECK_LAUNCH("mha_fwd");
    return GCGCN_OK;
}

// row-tiled tensor-core version for 65 <= max n <= 256 (gcn_stack_tiled.cu)
bool mha_bwd_tiled_usable(const gcgcn_batch* bt, int heads);
int launch_mha_bwd_tiled(const gcgcn_batch* bt, int heads, const float* q, const float* dS, float* dq, cudaStream_t st);

int launch_mha_bwd(const gcgcn_batch* bt, int heads, const float* q, const float* dS, float* dq,
                   cudaStream_t st) {
    if (bt->num_docs == 0) return GCGCN_OK;
    if (mha_bwd_tiled_usable(bt, heads)) return launch_mha_bwd_tiled(bt, heads, q, dS, dq, st);
    const int dh = D / heads;
    const float scale = 1.0f / sqrtf(static_cast<float>(dh));
    const size_t smem = mha_smem(bt->max_nodes, dh);
    dim3 grid(bt->num_docs, heads);
    const long long* pp = reinterpret_cast<const long long*>(bt->pair_ptr);
#define GCGCN_MHA_BWD(DH)                                                                         \
    case DH:                                                                                      \
        GCGCN_TRY(set_smem(mha_bwd_kernel<DH>, smem, "mha_bwd"));                                 \
        mha_bwd_kernel<DH><<<grid, MHA_THREADS, smem, st>>>(bt->node_ptr, pp, q, dS, dq,          \
                                                            bt->total_pairs, scale);              \
        break;
    switch (dh) {
        GCGCN_MHA_BWD(8)
        GCGCN_MHA_BWD(16)
        GCGCN_MHA_BWD(32)
        default:
            return fail(GCGCN_ERR_UNSUPPORTED, "head_num %d (d_h = %d) not supported; use 4, 8 or 16",
                        heads, dh);
    }
#undef GCGCN_MHA_BWD
    GCGCN_CHECK_LAUNCH("mha_bwd");
    return GCGCN_OK;
}

}  // namespace gcgcn
