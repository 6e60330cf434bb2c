// Dense fp32 projection C = alpha * op(A) op(B) + beta * C (+ bias), row-major, any strides.
//
// These are the only genuinely dense contractions on the path once the edge einsum is collapsed
// (SURVEY.md section 8a): node rows of the whole batch x [128 x 128*(1+H)] projection matrices in
// the forward pass, the transposed products for dX, and the K = (all node rows) reductions for
// the weight gradients.  This file holds the CUDA-core kernel (64x64x16 tiles, 4x4 register
// blocking, deterministic split-K); gemm_tc.cu runs every product with K >= 1 and M*N*K >= 2e6 on
// the tcgen05/TMEM kernels, so this one serves the smaller products and K = 0.
#include "common.cuh"

namespace gcgcn {

constexpr int GM = 64, GN = 64, GK = 16, GEMM_THREADS = 256;
constexpr int LDS_A = GM + 4, LDS_B = GN + 4;

template <bool TA, bool TB>
__global__ void __launch_bounds__(GEMM_THREADS)
gemm_kernel(int M, int N, int K, float alpha, const float* __restrict__ A, int lda,
            const float* __restrict__ B, int ldb, float beta, float* __restrict__ C, int ldc,
            const float* __restrict__ bias, float* __restrict__ partial, int k_per_split) {
    __shared__ __align__(16) float As[2][GK * LDS_A];  // As[k][m]
    __shared__ __align__(16) float Bs[2][GK * LDS_B];  // Bs[k][n]
    const int m0 = blockIdx.y * GM, n0 = blockIdx.x * GN;
    const int kbeg = blockIdx.z * k_per_split;
    const int kend = min(K, kbeg + k_per_split);
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;

    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    // element (m, k) of op(A) and (k, n) of op(B)
    auto a_at = [&](int m, int k) -> float {
        if (m >= M || k >= kend) return 0.f;
        return TA ? A[static_cast<size_t>(k) * lda + m] : A[static_cast<size_t>(m) * lda + k];
    };
    auto b_at = [&](int k, int n) -> float {
        if (n >= N || k >= kend) return 0.f;
        return TB ? B[static_cast<size_t>(n) * ldb + k] : B[static_cast<size_t>(k) * ldb + n];
    };
    const bool a_vec = (lda % 4 == 0) && ((reinterpret_cast<uintptr_t>(A) & 15) == 0) &&
                       (TA ? (m0 + GM <= M) : true);
    const bool b_vec = (ldb % 4 == 0) && ((reinterpret_cast<uintptr_t>(B) & 15) == 0) &&
                       (TB ? true : (n0 + GN <= N));

    auto load_tiles = [&](int buf, int k0) {
        float* as = As[buf];
        float* bs = Bs[buf];
        if (TA) {  // A stored [K][M]: rows of k are contiguous in m
            const int k = tid >> 4, m4 = (tid & 15) * 4;
            if (a_vec && k0 + k < kend) {
                float4 v = *reinterpret_cast<const float4*>(A + static_cast<size_t>(k0 + k) * lda + m0 + m4);
                *reinterpret_cast<float4*>(as + k * LDS_A + m4) = v;
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q) as[k * LDS_A + m4 + q] = a_at(m0 + m4 + q, k0 + k);
            }
        } else {   // A stored [M][K]: rows of m are contiguous in k -> transpose into As[k][m]
            const int m = tid >> 2, k4 = (tid & 3) * 4;
            float v[4];
            if (a_vec && m0 + m < M && k0 + k4 + 4 <= kend) {
                float4 t = *reinterpret_cast<const float4*>(A + static_cast<size_t>(m0 + m) * lda + k0 + k4);
                v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q) v[q] = a_at(m0 + m, k0 + k4 + q);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) as[(k4 + q) * LDS_A + m] = v[q];
        }
        if (!TB) {  // B stored [K][N]
            const int k = tid >> 4, n4 = (tid & 15) * 4;
            if (b_vec && k0 + k < kend) {
                float4 v = *reinterpret_cast<const float4*>(B + static_cast<size_t>(k0 + k) * ldb + n0 + n4);
                *reinterpret_cast<float4*>(bs + k * LDS_B + n4) = v;
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q) bs[k * LDS_B + n4 + q] = b_at(k0 + k, n0 + n4 + q);
            }
        } else {    // B stored [N][K] -> transpose into Bs[k][n]
            const int n = tid >> 2, k4 = (tid & 3) * 4;
            float v[4];
            if (b_vec && n0 + n < N && k0 + k4 + 4 <= kend) {
                float4 t = *reinterpret_cast<const float4*>(B + static_cast<size_t>(n0 + n) * ldb + k0 + k4);
                v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q) v[q] = b_at(k0 + k4 + q, n0 + n);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) bs[(k4 + q) * LDS_B + n] = v[q];
        }
    };

    int buf = 0;
    if (kbeg < kend) load_tiles(0, kbeg);
    __syncthreads();
    for (int k0 = kbeg; k0 < kend; k0 += GK) {
        if (k0 + GK < kend) load_tiles(buf ^ 1, k0 + GK);
        const float* as = As[buf];
        const float* bs = Bs[buf];
#pragma unroll
        for (int k = 0; k < GK; ++k) {
            const float4 a = *reinterpret_cast<const float4*>(as + k * LDS_A + ty * 4);
            const float4 b = *reinterpret_cast<const float4*>(bs + k * LDS_B + tx * 4);
            const float av[4] = {a.x, a.y, a.z, a.w};
            const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
        buf ^= 1;
    }

#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n >= N) continue;
            if (partial != nullptr) {
                partial[(static_cast<size_t>(blockIdx.z) * M + m) * N + n] = acc[i][j];
            } else {
                float v = alpha * acc[i][j];
                if (bias != nullptr) v += bias[n];
                float* c = C + static_cast<size_t>(m) * ldc + n;
                if (beta != 0.f) v += beta * (*c);
                *c = v;
            }
        }
    }
}

__global__ void __launch_bounds__(256)
splitk_reduce_kernel(const float* __restrict__ partial, int splits, int M, int N, float alpha, float beta,
                     float* __restrict__ C, int ldc, const float* __restrict__ bias, long long batch_stride_c) {
    const size_t idx = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const size_t total = static_cast<size_t>(M) * N;
    if (idx >= total) return;
    partial += static_cast<size_t>(blockIdx.y) * splits * total;      // batched: one product per blockIdx.y
    C += static_cast<size_t>(blockIdx.y) * batch_stride_c;
    // four interleaved partial sums in a fixed order (deterministic, 4 loads in flight)
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    int p = 0;
    for (; p + 4 <= splits; p += 4) {
        s0 += partial[(p + 0) * total + idx];
        s1 += partial[(p + 1) * total + idx];
        s2 += partial[(p + 2) * total + idx];
        s3 += partial[(p + 3) * total + idx];
    }
    for (; p < splits; ++p) s0 += partial[p * total + idx];
    const float s = (s0 + s1) + (s2 + s3);
    const int m = static_cast<int>(idx / N), n = static_cast<int>(idx - static_cast<size_t>(m) * N);
    float v = alpha * s;
    if (bias != nullptr) v += bias[n];
    float* c = C + static_cast<size_t>(m) * ldc + n;
    if (beta != 0.f) v += beta * (*c);
    *c = v;
}

// same, four consecutive columns per thread (N, ldc multiples of 4)
__global__ void __launch_bounds__(256)
splitk_reduce4_kernel(const float* __restrict__ partial, int splits, int M, int N, float alpha, float beta,
                      float* __restrict__ C, int ldc, const float* __restrict__ bias, long long batch_stride_c) {
    const size_t idx = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;    // float4 index
    const size_t total4 = static_cast<size_t>(M) * N / 4;
    if (idx >= total4) return;
    const float4* part = reinterpret_cast<const float4*>(partial) + static_cast<size_t>(blockIdx.y) * splits * total4;
    C += static_cast<size_t>(blockIdx.y) * batch_stride_c;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
    int p = 0;
    for (; p + 2 <= splits; p += 2) {
        const float4 u = part[(p + 0) * total4 + idx], w = part[(p + 1) * total4 + idx];
        a.x += u.x; a.y += u.y; a.z += u.z; a.w += u.w;
        b.x += w.x; b.y += w.y; b.z += w.z; b.w += w.w;
    }
    if (p < splits) {
        const float4 u = part[p * total4 + idx];
        a.x += u.x; a.y += u.y; a.z += u.z; a.w += u.w;
    }
    const int m = static_cast<int>(idx / (N / 4)), n = static_cast<int>(idx - static_cast<size_t>(m) * (N / 4)) * 4;
    float4 v = make_float4(alpha * (a.x + b.x), alpha * (a.y + b.y), alpha * (a.z + b.z), alpha * (a.w + b.w));
    if (bias != nullptr) {
        const float4 bb = *reinterpret_cast<const float4*>(bias + n);
        v.x += bb.x; v.y += bb.y; v.z += bb.z; v.w += bb.w;
    }
    float4* c = reinterpret_cast<float4*>(C + static_cast<size_t>(m) * ldc + n);
    if (beta != 0.f) {
        const float4 cur = *c;
        v.x += beta * cur.x; v.y += beta * cur.y; v.z += beta * cur.z; v.w += beta * cur.w;
    }
    *c = v;
}

// few outputs, many partials (weight gradients: one 128 x 128 tile split ~144 ways): 32 float4 columns x 8 split
// lanes per block so that a 16 K-element reduction runs on 128 blocks instead of 16; the 8 lane sums are
// combined in lane order (deterministic)
__global__ void __launch_bounds__(256)
splitk_reduce4_wide_kernel(const float* __restrict__ partial, int splits, int M, int N, float alpha, float beta,
                           float* __restrict__ C, int ldc, const float* __restrict__ bias, long long batch_stride_c) {
    __shared__ float4 sm[8][32];
    const int cx = threadIdx.x & 31, sy = threadIdx.x >> 5;
    const size_t idx = static_cast<size_t>(blockIdx.x) * 32 + cx;
    const size_t total4 = static_cast<size_t>(M) * N / 4;
    const float4* part = reinterpret_cast<const float4*>(partial) + static_cast<size_t>(blockIdx.y) * splits * total4;
    C += static_cast<size_t>(blockIdx.y) * batch_stride_c;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    if (idx < total4) {
#pragma unroll 4
        for (int p = sy; p < splits; p += 8) {
            const float4 u = part[static_cast<size_t>(p) * total4 + idx];
            a.x += u.x; a.y += u.y; a.z += u.z; a.w += u.w;
        }
    }
    sm[sy][cx] = a;
    __syncthreads();
    if (sy != 0 || idx >= total4) return;
#pragma unroll
    for (int y = 1; y < 8; ++y) {
        const float4 u = sm[y][cx];
        a.x += u.x; a.y += u.y; a.z += u.z; a.w += u.w;
    }
    const int m = static_cast<int>(idx / (N / 4)), n = static_cast<int>(idx - static_cast<size_t>(m) * (N / 4)) * 4;
    float4 v = make_float4(alpha * a.x, alpha * a.y, alpha * a.z, alpha * a.w);
    if (bias != nullptr) {
        const float4 bb = *reinterpret_cast<const float4*>(bias + n);
        v.x += bb.x; v.y += bb.y; v.z += bb.z; v.w += bb.w;
    }
    float4* c = reinterpret_cast<float4*>(C + static_cast<size_t>(m) * ldc + n);
    if (beta != 0.f) {
        const float4 cur = *c;
        v.x += beta * cur.x; v.y += beta * cur.y; v.z += beta * cur.z; v.w += beta * cur.w;
    }
    *c = v;
}

// column sums of a row-major [M, N] matrix (bias gradients), two deterministic stages
__global__ void __launch_bounds__(256)
colsum_partial_kernel(const float* __restrict__ X, int M, int N, int ldx, int rows_per_block,
                      float* __restrict__ partial) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= N) return;
    const int r0 = blockIdx.y * rows_per_block;
    const int r1 = min(M, r0 + rows_per_block);
    float s = 0.f;
    for (int r = r0; r < r1; ++r) s += X[static_cast<size_t>(r) * ldx + c];
    partial[static_cast<size_t>(blockIdx.y) * N + c] = s;
}

// N == 128 fast path: block = 32 float4 column lanes x 8 row lanes, fixed-order combine
__global__ void __launch_bounds__(256)
colsum128_partial_kernel(const float* __restrict__ X, int M, int ldx, int rows_per_block, float* __restrict__ partial) {
    __shared__ float4 red[8][32];
    const int cl = threadIdx.x & 31, rl = threadIdx.x >> 5;
    const int r0 = blockIdx.x * rows_per_block;
    const int r1 = min(M, r0 + rows_per_block);
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int r = r0 + rl; r < r1; r += 8) {
        const float4 v = *reinterpret_cast<const float4*>(X + static_cast<size_t>(r) * ldx + 4 * cl);
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    red[rl][cl] = s;
    __syncthreads();
    if (rl == 0) {
        float4 t = red[0][cl];
#pragma unroll
        for (int r = 1; r < 8; ++r) { const float4 v = red[r][cl]; t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w; }
        *reinterpret_cast<float4*>(partial + static_cast<size_t>(blockIdx.x) * 128 + 4 * cl) = t;
    }
}

int launch_reduce_partials(const float* partial, int parts, int width, float* out0, int width0,
                           float* out1, cudaStream_t st);

int launch_splitk_reduce(const float* partial, int splits, int M, int N, float alpha, float beta, float* C,
                         int ldc, const float* bias, cudaStream_t st, int batch = 1, long long sC = 0) {
    const size_t total = static_cast<size_t>(M) * N;
    const bool vec = N % 4 == 0 && ldc % 4 == 0 && sC % 4 == 0 && (reinterpret_cast<uintptr_t>(C) & 15) == 0 &&
                     (reinterpret_cast<uintptr_t>(partial) & 15) == 0 &&
                     (bias == nullptr || (reinterpret_cast<uintptr_t>(bias) & 15) == 0);
    if (vec && splits >= 16 && total / 4 <= 64 * 1024) {
        dim3 grid(ceil_div(total / 4, 32), batch);
        splitk_reduce4_wide_kernel<<<grid, 256, 0, st>>>(partial, splits, M, N, alpha, beta, C, ldc, bias, sC);
    } else if (vec) {
        dim3 grid(ceil_div(total / 4, 256), batch);
        splitk_reduce4_kernel<<<grid, 256, 0, st>>>(partial, splits, M, N, alpha, beta, C, ldc, bias, sC);
    } else {
        dim3 grid(ceil_div(total, 256), batch);
        splitk_reduce_kernel<<<grid, 256, 0, st>>>(partial, splits, M, N, alpha, beta, C, ldc, bias, sC);
    }
    GCGCN_CHECK_LAUNCH("splitk_reduce");
    return GCGCN_OK;
}

int launch_gemm_tc(int ta, int tb, int M, int N, int K, float alpha, const float* A, int lda, const float* B,
                   int ldb, float beta, float* C, int ldc, const float* bias, void* ws, size_t ws_bytes,
                   cudaStream_t st, int* taken, int batch, long long sA, long long sB, long long sC, void* pre_ws,
                   size_t pre_bytes, const float* bscale = nullptr, int lds = 0);

int launch_gemm(int ta, int tb, int M, int N, int K, float alpha, const float* A, int lda,
                const float* B, int ldb, float beta, float* C, int ldc, const float* bias, void* ws,
                size_t ws_bytes, cudaStream_t st) {
    if (M <= 0 || N <= 0) return GCGCN_OK;
    if (K < 0) return fail(GCGCN_ERR_INVALID_ARG, "gemm: K < 0");
    int taken = 0;
    GCGCN_TRY(launch_gemm_tc(ta, tb, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, bias, ws, ws_bytes, st, &taken,
                             1, 0, 0, 0, nullptr, 0));
    if (taken) return GCGCN_OK;
    const int tiles = ceil_div(M, GM) * ceil_div(N, GN);
    int splits = 1;
    const int target = 2 * sm_count();
    if (tiles < target && K >= 2048) {
        splits = min(ceil_div(target, tiles), ceil_div(K, 512));
        const size_t per = static_cast<size_t>(M) * N * sizeof(float);
        if (ws == nullptr || per == 0) splits = 1;
        else splits = static_cast<int>(std::min<size_t>(splits, ws_bytes / per));
        if (splits < 2) splits = 1;
    }
    int k_per = K;
    float* partial = nullptr;
    if (splits > 1) {
        k_per = ceil_div(ceil_div(K, splits), GK) * GK;
        splits = ceil_div(K, k_per);
        partial = static_cast<float*>(ws);
    }
    if (k_per == 0) k_per = GK;
    dim3 grid(ceil_div(N, GN), ceil_div(M, GM), splits);
#define GCGCN_GEMM(TA, TB)                                                                          \
    gemm_kernel<TA, TB><<<grid, GEMM_THREADS, 0, st>>>(M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, \
                                                       bias, partial, k_per)
    if (!ta && !tb) GCGCN_GEMM(false, false);
    else if (!ta && tb) GCGCN_GEMM(false, true);
    else if (ta && !tb) GCGCN_GEMM(true, false);
    else GCGCN_GEMM(true, true);
#undef GCGCN_GEMM
    timing_set_work(2.0 * M * N * K);
    GCGCN_CHECK_LAUNCH(ta ? (tb ? "gemm_tt" : "gemm_tn") : (tb ? "gemm_nt" : "gemm_nn"));
    if (splits > 1) GCGCN_TRY(launch_splitk_reduce(partial, splits, M, N, alpha, beta, C, ldc, bias, st));
    return GCGCN_OK;
}

// C[M, tiles * 128] (+)= A^T [M, K] x KR, column tile nt of KR being  scale[k][nt] * T[k][0..127]  (T a [K, 128] matrix):
// the weight gradient of a bilinear form, dW'[a][(r, b)] = sum_p h[p][a] dout[p][r] t[p][b], without materialising the
// [K, tiles * 128] operand.  Tensor-core path only (K >= 8192, M <= 256): GCGCN_ERR_UNSUPPORTED otherwise.
int launch_gemm_wgrad_scaled(int M, int tiles, int K, const float* A, int lda, const float* T, const float* scale, int lds,
                             float beta, float* C, int ldc, void* ws, size_t ws_bytes, cudaStream_t st, void* pre_ws,
                             size_t pre_bytes) {
    int taken = 0;
    GCGCN_TRY(launch_gemm_tc(1, 0, M, tiles * 128, K, 1.f, A, lda, T, 128, beta, C, ldc, nullptr, ws, ws_bytes, st, &taken, 1, 0,
                             0, 0, pre_ws, pre_bytes, scale, lds));
    if (!taken) return fail(GCGCN_ERR_UNSUPPORTED, "gemm_wgrad_scaled: shape not covered by the tensor-core path");
    return GCGCN_OK;
}

// `batch` independent products with the same shapes and strided operands (the per-head dense-connect
// weight gradients): one tensor-core launch when possible, else a loop over the single-product path
int launch_gemm_batched(int ta, int tb, int M, int N, int K, float alpha, const float* A, int lda, const float* B,
                        int ldb, float beta, float* C, int ldc, int batch, long long sA, long long sB, long long sC,
                        void* ws, size_t ws_bytes, cudaStream_t st) {
    if (M <= 0 || N <= 0 || batch <= 0) return GCGCN_OK;
    int taken = 0;
    GCGCN_TRY(launch_gemm_tc(ta, tb, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, nullptr, ws, ws_bytes, st, &taken,
                             batch, sA, sB, sC, nullptr, 0));
    if (taken) return GCGCN_OK;
    for (int b = 0; b < batch; ++b)
        GCGCN_TRY(launch_gemm(ta, tb, M, N, K, alpha, A + b * sA, lda, B + b * sB, ldb, beta, C + b * sC, ldc, nullptr,
                              ws, ws_bytes, st));
    return GCGCN_OK;
}

// out[c] = sum_r X[r, c]; ws holds the per-block partials
int launch_colsum(const float* X, int M, int N, int ldx, float* out, void* ws, size_t ws_bytes,
                  cudaStream_t st) {
    if (N <= 0) return GCGCN_OK;
    if (N == D && ldx % 4 == 0 && (reinterpret_cast<uintptr_t>(X) & 15) == 0 && M > 0) {
        const int rows_per_block = max(64, ceil_div(M, sm_count() * 4));
        const int parts = ceil_div(M, rows_per_block);
        if (ws == nullptr || ws_bytes < static_cast<size_t>(parts) * N * sizeof(float))
            return fail(GCGCN_ERR_WORKSPACE, "colsum: workspace too small");
        colsum128_partial_kernel<<<parts, 256, 0, st>>>(X, M, ldx, rows_per_block, static_cast<float*>(ws));
        GCGCN_CHECK_LAUNCH("colsum_partial");
        return launch_reduce_partials(static_cast<const float*>(ws), parts, N, out, N, nullptr, st);
    }
    int parts = max(1, min(ceil_div(M, 64), sm_count() * 16));
    const size_t need = static_cast<size_t>(parts) * N * sizeof(float);
    if (ws == nullptr || ws_bytes < need) return fail(GCGCN_ERR_WORKSPACE, "colsum: workspace too small");
    const int rows_per_block = max(1, ceil_div(M, parts));
    parts = max(1, ceil_div(M, rows_per_block));
    dim3 grid(ceil_div(N, 256), parts);
    colsum_partial_kernel<<<grid, 256, 0, st>>>(X, M, N, ldx, rows_per_block, static_cast<float*>(ws));
    GCGCN_CHECK_LAUNCH("colsum_partial");
    return launch_reduce_partials(static_cast<const float*>(ws), parts, N, out, N, nullptr, st);
}

}  // namespace gcgcn
