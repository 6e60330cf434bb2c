// Relation classifier and loss of GCGCN (SURVEY.md section 8f row 2, second half): the pieces around the dense
// products of  logits = Bilinear(128, 128, R)(h, t) + Linear(256, R)(cat[h, t])  (G:275-276, 356-358)  and the
// trainer's loss (config/Config.py:355-364).
//
// The bilinear form  out[p, r] = sum_{a,b} h[p,a] W[r,a,b] t[p,b]  is the one genuinely dense n^2-scale contraction of
// the model.  It runs on the tensor-memory GEMM of gemm_tc.cu (launch_gemm_rowop, launch_bilinear_wgrad) in fp32
// (3xTF32) or on bf16 operands, with W' = W viewed as [128, R*128]: the forward contracts each accumulator tile of h W'
// with t in the GEMM's epilogue, and the backward forms dh and dt the same way and generates the weight gradient's
// [pairs, R*128] operand from t and dout in the GEMM's producers, so that no [pairs, R*128] intermediate is ever stored.
// This file holds the kernels around them: the final transpose of the forward's partial sums, the per-document bias
// and the loss.
#include "common.cuh"

namespace gcgcn {

// ---- the trainer's loss (C:355-364): per document, mean over the ordered pairs i != j of BCELoss(sigmoid(z), y) ----
// torch's arithmetic: p = sigmoid(z); bce = (y - 1) max(log1p(-p), -100) - y max(log(p), -100)   (ATen Loss.cpp)
__device__ __forceinline__ float bce_of(float z, float y) {
    const float p = logit_sigmoid(z);
    return (y - 1.f) * fmaxf(log1pf(-p), -100.f) - y * fmaxf(logf(p), -100.f);
}
// d bce / d z = (p - y) / max((1 - p) p, 1e-12) * p (1 - p)      (binary_cross_entropy_backward, then sigmoid')
__device__ __forceinline__ float dbce_of(float z, float y) {
    const float p = logit_sigmoid(z);
    const float pq = (1.f - p) * p;
    return (p - y) / fmaxf(pq, 1e-12f) * pq;
}

// one CTA per document: pair_loss = mean_r bce; loss[b] = sum_{i != j} pair_loss / (n (n - 1)); fixed order
__global__ void __launch_bounds__(256)
pair_bce_fwd_kernel(const int* __restrict__ node_ptr, const long long* __restrict__ pair_ptr,
                    const float* __restrict__ z, const float* __restrict__ y, int R, float* __restrict__ loss) {
    __shared__ float red[8];
    const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = node_ptr[b + 1] - node_ptr[b];
    const long long p0 = pair_ptr[b];
    float acc = 0.f;
    for (int q = warp; q < n * n; q += 8) {
        const int i = q / n, j = q - i * n;
        if (i == j) continue;
        const float* zz = z + (p0 + q) * R;
        const float* yy = y + (p0 + q) * R;
        float s = 0.f;
        for (int r = lane; r < R; r += 32) s += bce_of(zz[r], yy[r]);
        s = warp_sum(s);
        acc += s / static_cast<float>(R);
    }
    if (lane == 0) red[warp] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int w = 0; w < 8; ++w) t += red[w];
        const int cnt = n * n - n;
        loss[b] = cnt > 0 ? t / static_cast<float>(cnt) : 0.f;
    }
}

__global__ void __launch_bounds__(256)
pair_bce_bwd_kernel(const int* __restrict__ node_ptr, const long long* __restrict__ pair_ptr,
                    const int* __restrict__ row_doc, const float* __restrict__ z, const float* __restrict__ y, int R,
                    const float* __restrict__ dloss, int total_nodes, float* __restrict__ dz) {
    // one warp per pair row (b, i): its n pairs are contiguous
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= total_nodes) return;
    const int b = row_doc[row];
    const int n = node_ptr[b + 1] - node_ptr[b], i = row - node_ptr[b];
    const float scale = n > 1 ? dloss[b] / (static_cast<float>(n * n - n) * static_cast<float>(R)) : 0.f;
    const long long base = (pair_ptr[b] + static_cast<long long>(i) * n) * R;
    const int cells = n * R;
    for (int c = lane; c < cells; c += 32) {
        const int j = c / R;
        dz[base + c] = (j == i) ? 0.f : scale * dbce_of(z[base + c], y[base + c]);
    }
}

// out[p][r] (+)= part[(2 r) ld + p] + part[(2 r + 1) ld + p] + bias[r]: the two column halves the row-dot GEMM leaves per
// (pair, relation), transposed through shared memory so that both the reads (along p) and the writes (along r) coalesce
__global__ void __launch_bounds__(256)
bilinear_finish_kernel(const float* __restrict__ part, long long ld, const float* __restrict__ bias, int rows, int R,
                       int accumulate, float* __restrict__ out, int ldo) {
    __shared__ float tile[32][33];
    const int p0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;          // 8 warps
    for (int rr = ty; rr < 32; rr += 8) {
        const int r = r0 + rr, p = p0 + tx;
        float v = 0.f;
        if (r < R && p < rows) v = part[(2LL * r) * ld + p] + part[(2LL * r + 1) * ld + p];
        tile[rr][tx] = v;
    }
    __syncthreads();
    for (int pp = ty; pp < 32; pp += 8) {
        const int p = p0 + pp, r = r0 + tx;
        if (p < rows && r < R) {
            float v = tile[tx][pp] + (bias != nullptr ? bias[r] : 0.f);
            float* o = out + static_cast<size_t>(p) * ldo + r;
            if (accumulate) v += *o;
            *o = v;
        }
    }
}

// ---- per-document vector added to every pair of the document (the BERT variant's cls_feature, B:346-347) ----------
// fwd: z[p][r] += v[doc(p)][r];  bwd: dv[b][r] = sum over the n_b^2 pairs of document b of dz[p][r] (fixed order)
__global__ void __launch_bounds__(256)
doc_bias_fwd_kernel(const int* __restrict__ node_ptr, const long long* __restrict__ pair_ptr, const float* __restrict__ v,
                    int R, float* __restrict__ z) {
    const int b = blockIdx.x;
    const int n = node_ptr[b + 1] - node_ptr[b];
    const long long cells = static_cast<long long>(n) * n * R;
    float* zz = z + pair_ptr[b] * R;
    const float* vv = v + static_cast<size_t>(b) * R;
    for (long long c = threadIdx.x; c < cells; c += blockDim.x) zz[c] += vv[c % R];
}
__global__ void __launch_bounds__(256)
doc_bias_bwd_kernel(const int* __restrict__ node_ptr, const long long* __restrict__ pair_ptr, const float* __restrict__ dz,
                    int R, float* __restrict__ dv) {
    const int b = blockIdx.x;
    const int n = node_ptr[b + 1] - node_ptr[b];
    const long long pairs = static_cast<long long>(n) * n;
    const float* zz = dz + pair_ptr[b] * R;
    for (int r = threadIdx.x; r < R; r += blockDim.x) {
        float acc = 0.f;
        for (long long p = 0; p < pairs; ++p) acc += zz[p * R + r];
        dv[static_cast<size_t>(b) * R + r] = acc;
    }
}

static int cl_grid(long long warps) { return static_cast<int>((warps + 7) / 8); }

int launch_doc_bias_fwd(const gcgcn_batch* bt, const float* v, int R, float* z, cudaStream_t st) {
    if (bt->num_docs <= 0 || R <= 0) return GCGCN_OK;
    doc_bias_fwd_kernel<<<bt->num_docs, 256, 0, st>>>(bt->node_ptr, reinterpret_cast<const long long*>(bt->pair_ptr), v, R, z);
    GCGCN_CHECK_LAUNCH("doc_bias_fwd");
    return GCGCN_OK;
}
int launch_doc_bias_bwd(const gcgcn_batch* bt, const float* dz, int R, float* dv, cudaStream_t st) {
    if (bt->num_docs <= 0 || R <= 0) return GCGCN_OK;
    doc_bias_bwd_kernel<<<bt->num_docs, 128, 0, st>>>(bt->node_ptr, reinterpret_cast<const long long*>(bt->pair_ptr), dz, R, dv);
    GCGCN_CHECK_LAUNCH("doc_bias_bwd");
    return GCGCN_OK;
}

int launch_bilinear_finish(const float* part, long long ld, const float* bias, int rows, int R, int accumulate, float* out,
                           int ldo, cudaStream_t st) {
    if (rows <= 0 || R <= 0) return GCGCN_OK;
    dim3 grid((rows + 31) / 32, (R + 31) / 32);
    bilinear_finish_kernel<<<grid, 256, 0, st>>>(part, ld, bias, rows, R, accumulate, out, ldo);
    GCGCN_CHECK_LAUNCH("bilinear_finish");
    return GCGCN_OK;
}

int launch_pair_bce_fwd(const gcgcn_batch* bt, const float* z, const float* y, int R, float* loss, cudaStream_t st) {
    if (bt->num_docs <= 0) return GCGCN_OK;
    pair_bce_fwd_kernel<<<bt->num_docs, 256, 0, st>>>(bt->node_ptr, reinterpret_cast<const long long*>(bt->pair_ptr), z, y,
                                                     R, loss);
    GCGCN_CHECK_LAUNCH("pair_bce_fwd");
    return GCGCN_OK;
}
int launch_pair_bce_bwd(const gcgcn_batch* bt, const float* z, const float* y, int R, const float* dloss, float* dz,
                        cudaStream_t st) {
    if (bt->total_nodes <= 0) return GCGCN_OK;
    pair_bce_bwd_kernel<<<cl_grid(bt->total_nodes), 256, 0, st>>>(bt->node_ptr,
                                                                 reinterpret_cast<const long long*>(bt->pair_ptr),
                                                                 bt->row_doc, z, y, R, dloss, bt->total_nodes, dz);
    GCGCN_CHECK_LAUNCH("pair_bce_bwd");
    return GCGCN_OK;
}

}  // namespace gcgcn
