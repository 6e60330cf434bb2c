// Edge-feature producer of GCGCN (SURVEY.md section 8f row 1): WordAttention + SentenceAttention (G:171-214) as
// the in-loop code uses them (G:299-327), restricted to what can reach the output.
//
// What the reference computes per hop and document is dense: [n, n, S, L, 128] expanded views pushed through
// three linears, a softmax over L and a relu-weighted sum over S.  What the output depends on is much less:
//   * attention_sent(context_before_att) is the same [L, 128] matrix SF for every (i, j, s) (G:179, 300) and
//     attention_pos(dis_embedding) has 21 distinct rows DF (G:180, 304-305), so the word scores are a table
//     T[l][k] = wa . tanh(SF[l] + DF[k]) + ba  -- 21 L values instead of n^2 S L;
//   * the sentence-level mask is ~sen_matrix[:, :, :, 0:1] (G:302): a slot survives only if its sentence contains
//     token 0; every other slot is masked to -1e5 before a RELU (G:209-212), contributes exactly 0 and passes
//     exactly zero gradient.  Only "active" slots (listed by the host from the wire format) are evaluated;
//   * a pair without active slots gets context_sent_att = linear_sentence_att.bias exactly.
// The kernels below are the non-GEMM pieces; the five small linears run on gcgcn_gemm.  Everything is
// deterministic (no atomics): scatters are written as gathers over host-built CSR tables.
//
//   word_table     T[a][k]                                   one warp per active token
//   word_pool      softmax over the sentence tokens of T[.][bucket(l)] (G:186-187), weighted ctx sum (G:188)
//   sent_pool      relu(va . tanh(Vs cw + Vp x_{j|i}) + ca)-weighted sum over a pair's active slots / (sent_num + 1e-10)
//   edge_fill      e[p] = b_ls (+ rows of the active pairs)
#include "common.cuh"

namespace gcgcn {

constexpr int EF_BUCKETS = 21;                 // config/Config.py:118 dis_num

__device__ __forceinline__ int ef_dis_bucket(int d) { return d == 0 ? 0 : min(10, 32 - __clz(d)); }
// dis_plus + signed log-bucket of token k against the mention span [a, b] (C:187-205, same rule as featurize.cu)
__device__ __forceinline__ int ef_pos_index(int k, int a, int b, int dis_plus) {
    if (k < a) return dis_plus - ef_dis_bucket(a - k);
    if (k > b) return dis_plus + ef_dis_bucket(k - b);
    return dis_plus;
}
__device__ __forceinline__ float dot4(const float4 a, const float4 b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
// tanh(x) = 1 - 2 / (exp(2x) + 1) on the fast exponential: |error| < 3e-7 over the whole range (saturation handled
// by the clamp), a third of the instructions of tanhf; the word table evaluates it
// 21 x 128 times per active token, forward and backward
__device__ __forceinline__ float ef_tanh(float x) {
    x = fminf(fmaxf(x, -20.f), 20.f);               // tanh(+-20) is +-1 in fp32; keeps exp finite for the fast divide
    return 1.0f - __fdividef(2.0f, __expf(2.0f * x) + 1.0f);
}
__device__ __forceinline__ float4 tanh4(float4 a, float4 b) {
    return make_float4(ef_tanh(a.x + b.x), ef_tanh(a.y + b.y), ef_tanh(a.z + b.z), ef_tanh(a.w + b.w));
}

// ---- word table -------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
word_table_fwd_kernel(const float* __restrict__ SF, const float* __restrict__ DF, const float* __restrict__ wa,
                      const float* __restrict__ ba, int tokens, float* __restrict__ T) {
    const int lane = threadIdx.x & 31;
    const int a = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (a >= tokens) return;
    const float4 sf = ld4(SF + static_cast<size_t>(a) * D + 4 * lane);
    const float4 w = ld4(wa + 4 * lane);
    const float b = ba[0];
#pragma unroll 3
    for (int k = 0; k < EF_BUCKETS; ++k) {
        const float4 th = tanh4(sf, ld4(DF + k * D + 4 * lane));
        const float s = warp_sum(dot4(w, th));
        if (lane == 0) T[static_cast<size_t>(a) * EF_BUCKETS + k] = s + b;
    }
}

constexpr int WT_PARTIAL = EF_BUCKETS * D + D + 4;       // dDF [21][128], dwa [128], dba + 3 pad (rows stay 16-byte aligned)

// dSF[a] = sum_k dT[a][k] wa (1 - th^2);  per-warp partial sums of dDF[k], dwa, dba (reduced by reduce_partials)
__global__ void __launch_bounds__(128)
word_table_bwd_kernel(const float* __restrict__ SF, const float* __restrict__ DF, const float* __restrict__ wa,
                      const float* __restrict__ dT, int tokens, float* __restrict__ dSF, float* __restrict__ partial) {
    const int lane = threadIdx.x & 31;
    const int gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int nw = gridDim.x * (blockDim.x >> 5);
    const float4 w = ld4(wa + 4 * lane);
    float4 accDF[EF_BUCKETS];
#pragma unroll
    for (int k = 0; k < EF_BUCKETS; ++k) accDF[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 accw = make_float4(0.f, 0.f, 0.f, 0.f);
    float accb = 0.f;
    for (int a = gw; a < tokens; a += nw) {
        const float4 sf = ld4(SF + static_cast<size_t>(a) * D + 4 * lane);
        float4 dsf = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int k = 0; k < EF_BUCKETS; ++k) {
            const float s = dT[static_cast<size_t>(a) * EF_BUCKETS + k];
            const float4 th = tanh4(sf, ld4(DF + k * D + 4 * lane));
            float4 dp;
            dp.x = s * w.x * (1.f - th.x * th.x); dp.y = s * w.y * (1.f - th.y * th.y);
            dp.z = s * w.z * (1.f - th.z * th.z); dp.w = s * w.w * (1.f - th.w * th.w);
            dsf.x += dp.x; dsf.y += dp.y; dsf.z += dp.z; dsf.w += dp.w;
            accDF[k].x += dp.x; accDF[k].y += dp.y; accDF[k].z += dp.z; accDF[k].w += dp.w;
            accw.x += s * th.x; accw.y += s * th.y; accw.z += s * th.z; accw.w += s * th.w;
            accb += s;
        }
        st4(dSF + static_cast<size_t>(a) * D + 4 * lane, dsf);
    }
    float* out = partial + static_cast<size_t>(gw) * WT_PARTIAL;
#pragma unroll
    for (int k = 0; k < EF_BUCKETS; ++k) st4(out + k * D + 4 * lane, accDF[k]);
    st4(out + EF_BUCKETS * D + 4 * lane, accw);
    if (lane < 4) out[EF_BUCKETS * D + D + lane] = lane == 0 ? accb : 0.f;
}

// ---- word-level attention over the tokens of one active slot ----------------------------------------------
struct EdgeTabs {
    int tokens, slots, pairs, att_total, dis_plus;
    const int* tok_first;      // [tokens] index of token 0 of the same document among the active tokens
    const int* tok_slot_lo;    // [tokens] first active slot of the token's document
    const int* tok_slot_hi;    // [tokens] one past its last
    const int* slot_tok0;      // [slots]
    const int* slot_len;       // [slots] sentence tokens [0, len)
    const int* slot_span;      // [slots][4] h0, h1, t0, t1
    const int* slot_att;       // [slots] offset of the slot's 2 * len attention entries (h side, then t side)
    const int* slot_rowi;      // [slots] global node row of the pair's row entity i
    const int* slot_rowj;      // [slots] ... of its column entity j
    const long long* pair_idx; // [pairs] global pair index of the active pair
    const int* pair_slot_ptr;  // [pairs + 1] its slots (slots are sorted by pair)
    const float* pair_denom;   // [pairs] float32(sent_num) + 1e-10  (G:206, 213)
    const int* node_ctr_ptr;   // [total_nodes + 1] contributions (slot * 2 + side) whose node embedding is this row
    const int* node_ctr;
    int adocs, max_len;        // documents with at least one active slot; their longest first sentence
    const int* adoc_tok0;      // [adocs] active-token index of the document's token 0
    const int* adoc_len;       // [adocs] active tokens of the document
    const int* adoc_slot_lo;   // [adocs] its active slots [lo, hi)
    const int* adoc_slot_hi;
};

__global__ void __launch_bounds__(256)
word_pool_fwd_kernel(const EdgeTabs tb, const float* __restrict__ T, const float* __restrict__ ctx,
                     float* __restrict__ att, float* __restrict__ cwa) {
    const int lane = threadIdx.x & 31;
    const int u = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);      // (slot, side)
    if (u >= 2 * tb.slots) return;
    const int s = u >> 1, side = u & 1;
    const int len = tb.slot_len[s], a0 = tb.slot_tok0[s];
    const int m0 = tb.slot_span[4 * s + 2 * side], m1 = tb.slot_span[4 * s + 2 * side + 1];
    float* at = att + tb.slot_att[s] + side * len;
    float mx = -INFINITY;
    for (int l = lane; l < len; l += 32) {
        const float v = T[static_cast<size_t>(a0 + l) * EF_BUCKETS + ef_pos_index(l, m0, m1, tb.dis_plus)];
        at[l] = v;
        mx = fmaxf(mx, v);
    }
    mx = warp_max(mx);
    float sum = 0.f;
    for (int l = lane; l < len; l += 32) {
        const float e = expf(at[l] - mx);
        at[l] = e;
        sum += e;
    }
    sum = warp_sum(sum);
    const float inv = 1.0f / sum;
    for (int l = lane; l < len; l += 32) at[l] *= inv;
    __syncwarp();
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    const float* crow = ctx + static_cast<size_t>(a0) * D + 4 * lane;
    for (int l = 0; l < len; l += 8) {                  // eight context rows in flight per lane (the loop is latency bound)
        float4 r[8];
        float w[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const bool ok = l + u < len;
            r[u] = ok ? ld4(crow + static_cast<size_t>(l + u) * D) : make_float4(0.f, 0.f, 0.f, 0.f);
            w[u] = ok ? at[l + u] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            acc.x += w[u] * r[u].x; acc.y += w[u] * r[u].y; acc.z += w[u] * r[u].z; acc.w += w[u] * r[u].w;
        }
    }
    st4(cwa + static_cast<size_t>(s) * 2 * D + side * D + 4 * lane, acc);
}

// dlog[l] = att[l] (g[l] - sum_l att g),  g[l] = dcwa . ctx[l]
__global__ void __launch_bounds__(256)
word_pool_bwd_logit_kernel(const EdgeTabs tb, const float* __restrict__ ctx, const float* __restrict__ att,
                           const float* __restrict__ dcwa, float* __restrict__ dlog) {
    const int lane = threadIdx.x & 31;
    const int u = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (u >= 2 * tb.slots) return;
    const int s = u >> 1, side = u & 1;
    const int len = tb.slot_len[s], a0 = tb.slot_tok0[s];
    const float* at = att + tb.slot_att[s] + side * len;
    float* dl = dlog + tb.slot_att[s] + side * len;
    const float4 dc = ld4(dcwa + static_cast<size_t>(s) * 2 * D + side * D + 4 * lane);
    float dot = 0.f;
    const float* crow = ctx + static_cast<size_t>(a0) * D + 4 * lane;
    for (int l = 0; l < len; l += 8) {                  // eight context rows in flight, then eight independent reductions
        float p[8];
#pragma unroll
        for (int u = 0; u < 8; ++u)
            p[u] = l + u < len ? dot4(dc, ld4(crow + static_cast<size_t>(l + u) * D)) : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
            for (int u = 0; u < 8; ++u) p[u] += __shfl_xor_sync(0xffffffffu, p[u], o);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            if (l + u < len) {
                if (lane == 0) dl[l + u] = p[u];
                dot += at[l + u] * p[u];
            }
        }
    }
    __syncwarp();
    for (int l = lane; l < len; l += 32) dl[l] = at[l] * (dl[l] - dot);
}

// per active token: dctx[a] = sum over the document's (slot, side) covering it of att * dcwa,
//                   dT[a][k] = sum over those with bucket == k of dlog
__global__ void __launch_bounds__(256)
word_pool_bwd_token_kernel(const EdgeTabs tb, const float* __restrict__ att, const float* __restrict__ dlog,
                           const float* __restrict__ dcwa, float* __restrict__ dctx, float* __restrict__ dT) {
    const int lane = threadIdx.x & 31;
    const int a = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (a >= tb.tokens) return;
    const int l = a - tb.tok_first[a];
    const int lo = tb.tok_slot_lo[a], hi = tb.tok_slot_hi[a];
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int s0 = lo; s0 < hi; s0 += 4) {               // four slots (eight gradient rows) in flight per lane
        float4 d[8];
        float w[8];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int s = s0 + u;
            const int len = s < hi ? tb.slot_len[s] : 0;
            const bool ok = l < len;
            const int off = ok ? tb.slot_att[s] : 0;
#pragma unroll
            for (int side = 0; side < 2; ++side) {
                w[2 * u + side] = ok ? att[off + side * len + l] : 0.f;
                d[2 * u + side] = ok ? ld4(dcwa + static_cast<size_t>(s) * 2 * D + side * D + 4 * lane)
                                     : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            acc.x += w[u] * d[u].x; acc.y += w[u] * d[u].y; acc.z += w[u] * d[u].z; acc.w += w[u] * d[u].w;
        }
    }
    st4(dctx + static_cast<size_t>(a) * D + 4 * lane, acc);
    // bins: lane k owns bucket k; entries (slot, side) are taken 32 at a time, one per lane
    float bin = 0.f;
    const int entries = 2 * (hi - lo);
    for (int e0 = 0; e0 < entries; e0 += 32) {
        const int e = e0 + lane;
        int k = -1;
        float v = 0.f;
        if (e < entries) {
            const int s = lo + (e >> 1), side = e & 1, len = tb.slot_len[s];
            if (l < len) {
                k = ef_pos_index(l, tb.slot_span[4 * s + 2 * side], tb.slot_span[4 * s + 2 * side + 1], tb.dis_plus);
                v = dlog[tb.slot_att[s] + side * len + l];
            }
        }
#pragma unroll
        for (int kk = 0; kk < EF_BUCKETS; ++kk) {
            const float t = warp_sum(k == kk ? v : 0.f);
            if (lane == kk) bin += t;
        }
    }
    if (lane < EF_BUCKETS) dT[static_cast<size_t>(a) * EF_BUCKETS + lane] = bin;
}

// ---- the same three kernels with one CTA per document and its first sentence in shared memory ----------------------
// Every (slot, side) of a document walks the same <= 96 context rows and every token of it the same gradient rows: read
// through L2 per warp (the kernels above) that is 30-40x redundant traffic and the L2 bandwidth becomes the limit
// (4 GB per launch at the bench shard).  Here the context tile is loaded once per document, the gradient rows once per
// chunk of 64 entries.  Used when the longest first sentence of the batch fits (WP_MAX_LEN tokens).
constexpr int WP_MAX_LEN = 96, WP_ENT = 32;

__global__ void __launch_bounds__(256)
word_pool_fwd_doc_kernel(const EdgeTabs tb, const float* __restrict__ T, const float* __restrict__ ctx,
                         float* __restrict__ att, float* __restrict__ cwa) {
    extern __shared__ __align__(16) float wp_smem[];
    const int d = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int a0 = tb.adoc_tok0[d], L = tb.adoc_len[d], lo = tb.adoc_slot_lo[d], hi = tb.adoc_slot_hi[d];
    float* ctx_s = wp_smem;                                   // [L][128]
    float* T_s = ctx_s + L * D;                               // [L][21] word-score table rows of the document
    for (int i = threadIdx.x; i < L * (D / 4); i += 256) st4(ctx_s + 4 * i, ld4(ctx + static_cast<size_t>(a0) * D + 4 * i));
    for (int i = threadIdx.x; i < L * EF_BUCKETS; i += 256) T_s[i] = T[static_cast<size_t>(a0) * EF_BUCKETS + i];
    __syncthreads();
    for (int u = warp; u < 2 * (hi - lo); u += 8) {
        const int s = lo + (u >> 1), side = u & 1;
        const int len = tb.slot_len[s];
        const int m0 = tb.slot_span[4 * s + 2 * side], m1 = tb.slot_span[4 * s + 2 * side + 1];
        float* at = att + tb.slot_att[s] + side * len;
        // (len <= L <= 96: at most three logits per lane, kept in registers)
        float v[3];
        float mx = -INFINITY;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const int l = lane + 32 * r;
            v[r] = l < len ? T_s[l * EF_BUCKETS + ef_pos_index(l, m0, m1, tb.dis_plus)] : -INFINITY;
            mx = fmaxf(mx, v[r]);
        }
        mx = warp_max(mx);
        float sum = 0.f;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            v[r] = lane + 32 * r < len ? expf(v[r] - mx) : 0.f;
            sum += v[r];
        }
        sum = warp_sum(sum);
        const float inv = 1.0f / sum;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            v[r] *= inv;
            if (lane + 32 * r < len) at[lane + 32 * r] = v[r];
        }
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int l = 0; l < len; ++l) {
            const float w = __shfl_sync(0xffffffffu, l < 32 ? v[0] : (l < 64 ? v[1] : v[2]), l & 31);
            const float4 r = ld4(ctx_s + l * D + 4 * lane);
            acc.x += w * r.x; acc.y += w * r.y; acc.z += w * r.z; acc.w += w * r.w;
        }
        st4(cwa + static_cast<size_t>(s) * 2 * D + side * D + 4 * lane, acc);
    }
}

__global__ void __launch_bounds__(256)
word_pool_bwd_doc_kernel(const EdgeTabs tb, const float* __restrict__ ctx, const float* __restrict__ att,
                         const float* __restrict__ dcwa, float* __restrict__ dctx, float* __restrict__ dT) {
    extern __shared__ __align__(16) float wp_smem[];
    __shared__ int m_len[WP_ENT], m_off[WP_ENT], m_m0[WP_ENT], m_m1[WP_ENT];
    const int d = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int a0 = tb.adoc_tok0[d], L = tb.adoc_len[d], lo = tb.adoc_slot_lo[d], hi = tb.adoc_slot_hi[d];
    const int LP = L + 1;                                     // row stride of the per-entry token arrays (bank spread)
    float* ctx_s = wp_smem;                                   // [L][128]
    float* d_s = ctx_s + L * D;                               // [WP_ENT][128] gradient rows of the current chunk
    float* bin_s = d_s + WP_ENT * D;                          // [L][32] dT bins (column k = bucket k)
    float* at_s = bin_s + L * 32;                             // [WP_ENT][LP] attention weights (0 past the sentence)
    float* dl_s = at_s + WP_ENT * LP;                         // [WP_ENT][LP] d logits
    for (int i = threadIdx.x; i < L * (D / 4); i += 256) st4(ctx_s + 4 * i, ld4(ctx + static_cast<size_t>(a0) * D + 4 * i));
    for (int i = threadIdx.x; i < L * 32; i += 256) bin_s[i] = 0.f;
    const int E = 2 * (hi - lo);
    for (int e0 = 0; e0 < E; e0 += WP_ENT) {
        const int en = min(WP_ENT, E - e0);
        __syncthreads();                                      // previous chunk fully consumed (and the tile loads above done)
        if (threadIdx.x < en) {
            const int e = e0 + threadIdx.x, s = lo + (e >> 1), side = e & 1, len = tb.slot_len[s];
            m_len[threadIdx.x] = len;
            m_off[threadIdx.x] = tb.slot_att[s] + side * len;
            m_m0[threadIdx.x] = tb.slot_span[4 * s + 2 * side];
            m_m1[threadIdx.x] = tb.slot_span[4 * s + 2 * side + 1];
        }
        for (int i = threadIdx.x; i < en * (D / 4); i += 256) {
            const int j = i / (D / 4), q = i % (D / 4), e = e0 + j;
            st4(d_s + j * D + 4 * q, ld4(dcwa + static_cast<size_t>(lo + (e >> 1)) * 2 * D + (e & 1) * D + 4 * q));
        }
        __syncthreads();
        for (int i = threadIdx.x; i < en * L; i += 256) {
            const int j = i / L, l = i - j * L;
            at_s[j * LP + l] = l < m_len[j] ? att[m_off[j] + l] : 0.f;
        }
        __syncthreads();
        // (a) dlog[l] = att[l] (g[l] - sum_l att g), g[l] = dcwa . ctx[l]
        for (int j = warp; j < en; j += 8) {
            const int len = m_len[j];
            const float4 dc = ld4(d_s + j * D + 4 * lane);
            float dot = 0.f;
            for (int l = 0; l < len; l += 4) {
                float p[4];
#pragma unroll
                for (int v = 0; v < 4; ++v) p[v] = l + v < len ? dot4(dc, ld4(ctx_s + (l + v) * D + 4 * lane)) : 0.f;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
                    for (int v = 0; v < 4; ++v) p[v] += __shfl_xor_sync(0xffffffffu, p[v], o);
                }
#pragma unroll
                for (int v = 0; v < 4; ++v) {
                    if (l + v < len) {
                        if (lane == 0) dl_s[j * LP + l + v] = p[v];
                        dot += at_s[j * LP + l + v] * p[v];
                    }
                }
            }
            __syncwarp();
            for (int l = lane; l < L; l += 32) dl_s[j * LP + l] = l < len ? at_s[j * LP + l] * (dl_s[j * LP + l] - dot) : 0.f;
        }
        __syncthreads();
        // (b) per token: dctx = sum over the entries covering it of att * dcwa;  dT bins of dlog by position bucket
        for (int l = warp; l < L; l += 8) {
            float w = 0.f, v = 0.f;
            int k = -1;
            if (lane < en && l < m_len[lane]) {
                w = at_s[lane * LP + l];
                v = dl_s[lane * LP + l];
                k = ef_pos_index(l, m_m0[lane], m_m1[lane], tb.dis_plus);
            }
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int jj = 0; jj < en; ++jj) {                 // entries in order: a fixed summation order
                const float wj = __shfl_sync(0xffffffffu, w, jj);
                const float4 r = ld4(d_s + jj * D + 4 * lane);
                acc.x += wj * r.x; acc.y += wj * r.y; acc.z += wj * r.z; acc.w += wj * r.w;
            }
            float bin = 0.f;
#pragma unroll
            for (int kk = 0; kk < EF_BUCKETS; ++kk) {
                const float t = warp_sum(k == kk ? v : 0.f);
                if (lane == kk) bin = t;
            }
            float* o = dctx + static_cast<size_t>(a0 + l) * D + 4 * lane;
            if (e0 > 0) {
                const float4 old = ld4(o);
                acc.x += old.x; acc.y += old.y; acc.z += old.z; acc.w += old.w;
            }
            st4(o, acc);
            bin_s[l * 32 + lane] += bin;
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < L * EF_BUCKETS; i += 256) {
        const int l = i / EF_BUCKETS, k = i - l * EF_BUCKETS;
        dT[static_cast<size_t>(a0 + l) * EF_BUCKETS + k] = bin_s[l * 32 + k];
    }
}

// ---- sentence-level attention over the active slots of one pair -----------------------------------------
constexpr int SP_PARTIAL = D + 4;      // dva [128], dca + 3 pad

__global__ void __launch_bounds__(256)
sent_pool_fwd_kernel(const EdgeTabs tb, const float* __restrict__ cw, const float* __restrict__ sfeat,
                     const float* __restrict__ nfeat, const float* __restrict__ va, const float* __restrict__ ca,
                     float* __restrict__ score, float* __restrict__ csa) {
    const int lane = threadIdx.x & 31;
    const int p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (p >= tb.pairs) return;
    const float4 v = ld4(va + 4 * lane);
    const float c = ca[0];
    float4 ah = make_float4(0.f, 0.f, 0.f, 0.f), at = ah;
    for (int s = tb.pair_slot_ptr[p]; s < tb.pair_slot_ptr[p + 1]; ++s) {
        const float4 sf = ld4(sfeat + static_cast<size_t>(s) * D + 4 * lane);
        const float4 nj = ld4(nfeat + static_cast<size_t>(tb.slot_rowj[s]) * D + 4 * lane);   // "h" embeds the column entity (G:320)
        const float4 ni = ld4(nfeat + static_cast<size_t>(tb.slot_rowi[s]) * D + 4 * lane);   // "t" embeds the row entity (G:321)
        const float sh = warp_sum(dot4(v, tanh4(sf, nj))) + c;
        const float st_ = warp_sum(dot4(v, tanh4(sf, ni))) + c;
        if (lane == 0) { score[2 * s] = sh; score[2 * s + 1] = st_; }
        const float wh = fmaxf(sh, 0.f), wt = fmaxf(st_, 0.f);
        const float4 r = ld4(cw + static_cast<size_t>(s) * D + 4 * lane);
        ah.x += wh * r.x; ah.y += wh * r.y; ah.z += wh * r.z; ah.w += wh * r.w;
        at.x += wt * r.x; at.y += wt * r.y; at.z += wt * r.z; at.w += wt * r.w;
    }
    const float den = tb.pair_denom[p];
    ah.x /= den; ah.y /= den; ah.z /= den; ah.w /= den;
    at.x /= den; at.y /= den; at.z /= den; at.w /= den;
    st4(csa + static_cast<size_t>(p) * 2 * D + 4 * lane, ah);
    st4(csa + static_cast<size_t>(p) * 2 * D + D + 4 * lane, at);
}

__global__ void __launch_bounds__(128)
sent_pool_bwd_kernel(const EdgeTabs tb, const float* __restrict__ cw, const float* __restrict__ sfeat,
                     const float* __restrict__ nfeat, const float* __restrict__ va, const float* __restrict__ score,
                     const float* __restrict__ dcsa, float* __restrict__ dcw, float* __restrict__ dsfeat,
                     float* __restrict__ dpre, float* __restrict__ partial) {
    const int lane = threadIdx.x & 31;
    const int gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int nw = gridDim.x * (blockDim.x >> 5);
    const float4 v = ld4(va + 4 * lane);
    float4 accv = make_float4(0.f, 0.f, 0.f, 0.f);
    float accc = 0.f;
    for (int p = gw; p < tb.pairs; p += nw) {
        const float den = tb.pair_denom[p];
        const float4 dh = ld4(dcsa + static_cast<size_t>(p) * 2 * D + 4 * lane);
        const float4 dt = ld4(dcsa + static_cast<size_t>(p) * 2 * D + D + 4 * lane);
        for (int s = tb.pair_slot_ptr[p]; s < tb.pair_slot_ptr[p + 1]; ++s) {
            const float sh = score[2 * s], st_ = score[2 * s + 1];
            const float wh = fmaxf(sh, 0.f), wt = fmaxf(st_, 0.f);
            const float4 r = ld4(cw + static_cast<size_t>(s) * D + 4 * lane);
            float4 g;
            g.x = (wh * dh.x + wt * dt.x) / den; g.y = (wh * dh.y + wt * dt.y) / den;
            g.z = (wh * dh.z + wt * dt.z) / den; g.w = (wh * dh.w + wt * dt.w) / den;
            st4(dcw + static_cast<size_t>(s) * D + 4 * lane, g);
            const float dsh = sh > 0.f ? warp_sum(dot4(dh, r)) / den : 0.f;     // relu'(0) = 0 like torch
            const float dst = st_ > 0.f ? warp_sum(dot4(dt, r)) / den : 0.f;
            const float4 sf = ld4(sfeat + static_cast<size_t>(s) * D + 4 * lane);
            const float4 thh = tanh4(sf, ld4(nfeat + static_cast<size_t>(tb.slot_rowj[s]) * D + 4 * lane));
            const float4 tht = tanh4(sf, ld4(nfeat + static_cast<size_t>(tb.slot_rowi[s]) * D + 4 * lane));
            float4 ph, pt;
            ph.x = dsh * v.x * (1.f - thh.x * thh.x); ph.y = dsh * v.y * (1.f - thh.y * thh.y);
            ph.z = dsh * v.z * (1.f - thh.z * thh.z); ph.w = dsh * v.w * (1.f - thh.w * thh.w);
            pt.x = dst * v.x * (1.f - tht.x * tht.x); pt.y = dst * v.y * (1.f - tht.y * tht.y);
            pt.z = dst * v.z * (1.f - tht.z * tht.z); pt.w = dst * v.w * (1.f - tht.w * tht.w);
            st4(dpre + (static_cast<size_t>(s) * 2) * D + 4 * lane, ph);
            st4(dpre + (static_cast<size_t>(s) * 2 + 1) * D + 4 * lane, pt);
            st4(dsfeat + static_cast<size_t>(s) * D + 4 * lane, make_float4(ph.x + pt.x, ph.y + pt.y, ph.z + pt.z, ph.w + pt.w));
            accv.x += dsh * thh.x + dst * tht.x; accv.y += dsh * thh.y + dst * tht.y;
            accv.z += dsh * thh.z + dst * tht.z; accv.w += dsh * thh.w + dst * tht.w;
            accc += dsh + dst;
        }
    }
    float* out = partial + static_cast<size_t>(gw) * SP_PARTIAL;
    st4(out + 4 * lane, accv);
    if (lane < 4) out[D + lane] = lane == 0 ? accc : 0.f;
}

// dnfeat[r] = sum of dpre over the (slot, side) entries whose node embedding is row r (fixed order)
__global__ void __launch_bounds__(256)
node_collect_kernel(const int* __restrict__ ptr, const int* __restrict__ ctr, const float* __restrict__ dpre, int rows,
                    float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= rows) return;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int k = ptr[r]; k < ptr[r + 1]; ++k) {
        const float4 d = ld4(dpre + static_cast<size_t>(ctr[k]) * D + 4 * lane);
        acc.x += d.x; acc.y += d.y; acc.z += d.z; acc.w += d.w;
    }
    st4(out + static_cast<size_t>(r) * D + 4 * lane, acc);
}

// ---- e[p] = bias, + rows of the active pairs ---------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
edge_fill_kernel(const float* __restrict__ bias, long long total_pairs, T* __restrict__ e) {
    const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;     // float4 index
    if (idx >= total_pairs * (D / 4)) return;
    const float4 b = ld4(bias + 4 * (idx & (D / 4 - 1)));
    Vec4<T>::store(e + idx * 4, b);
}
template <typename T>
__global__ void __launch_bounds__(256)
edge_scatter_kernel(const float* __restrict__ bias, const float* __restrict__ rows, const long long* __restrict__ pair_idx,
                    int pairs, T* __restrict__ e) {
    const int lane = threadIdx.x & 31;
    const int p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (p >= pairs) return;
    const float4 b = ld4(bias + 4 * lane);
    const float4 r = ld4(rows + static_cast<size_t>(p) * D + 4 * lane);
    Vec4<T>::store(e + pair_idx[p] * D + 4 * lane, make_float4(r.x + b.x, r.y + b.y, r.z + b.z, r.w + b.w));
}
template <typename T>
__global__ void __launch_bounds__(256)
edge_gather_kernel(const T* __restrict__ de, const long long* __restrict__ pair_idx, int pairs, float* __restrict__ rows) {
    const int lane = threadIdx.x & 31;
    const int p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (p >= pairs) return;
    st4(rows + static_cast<size_t>(p) * D + 4 * lane, Vec4<T>::load(de + pair_idx[p] * D + 4 * lane));
}
// column sums of a [pairs, 128] edge tensor in either storage type: per-block partials, fixed order
template <typename T>
__global__ void __launch_bounds__(256)
edge_colsum_kernel(const T* __restrict__ de, long long total_pairs, long long rows_per_block, float* __restrict__ partial) {
    __shared__ float4 red[8][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long r0 = blockIdx.x * rows_per_block, r1 = min(total_pairs, r0 + rows_per_block);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (long long r = r0 + warp; r < r1; r += 8) {
        const float4 v = Vec4<T>::load(de + r * D + 4 * lane);
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    red[warp][lane] = acc;
    __syncthreads();
    if (warp == 0) {
        float4 t = red[0][lane];
        for (int w = 1; w < 8; ++w) { t.x += red[w][lane].x; t.y += red[w][lane].y; t.z += red[w][lane].z; t.w += red[w][lane].w; }
        st4(partial + static_cast<size_t>(blockIdx.x) * D + 4 * lane, t);
    }
}

int launch_reduce_partials(const float* partial, int parts, int width, float* out0, int width0, float* out1,
                           cudaStream_t st);

static EdgeTabs make_tabs(const gcgcn_edge_tables* t) {
    EdgeTabs tb;
    tb.tokens = t->num_tokens; tb.slots = t->num_slots; tb.pairs = t->num_pairs; tb.att_total = t->att_total;
    tb.dis_plus = t->dis_plus;
    tb.tok_first = t->tok_first; tb.tok_slot_lo = t->tok_slot_lo; tb.tok_slot_hi = t->tok_slot_hi;
    tb.slot_tok0 = t->slot_tok0; tb.slot_len = t->slot_len; tb.slot_span = t->slot_span; tb.slot_att = t->slot_att;
    tb.slot_rowi = t->slot_rowi; tb.slot_rowj = t->slot_rowj;
    tb.pair_idx = reinterpret_cast<const long long*>(t->pair_idx); tb.pair_slot_ptr = t->pair_slot_ptr;
    tb.pair_denom = t->pair_denom; tb.node_ctr_ptr = t->node_ctr_ptr; tb.node_ctr = t->node_ctr;
    tb.adocs = t->num_active_docs; tb.max_len = t->max_active_len;
    tb.adoc_tok0 = t->adoc_tok0; tb.adoc_len = t->adoc_len; tb.adoc_slot_lo = t->adoc_slot_lo; tb.adoc_slot_hi = t->adoc_slot_hi;
    return tb;
}

static int warps_grid(long long warps, int per_block) { return static_cast<int>((warps + per_block - 1) / per_block); }

int launch_word_table_fwd(const float* SF, const float* DF, const float* wa, const float* ba, int tokens, float* T,
                          cudaStream_t st) {
    if (tokens <= 0) return GCGCN_OK;
    word_table_fwd_kernel<<<warps_grid(tokens, 8), 256, 0, st>>>(SF, DF, wa, ba, tokens, T);
    GCGCN_CHECK_LAUNCH("word_table_fwd");
    return GCGCN_OK;
}

int word_table_parts(int tokens) { return std::max(1, std::min(sm_count() * 2, (tokens + 3) / 4)) * 4; }

// out: [21 * 128 + 128 + 4] = dDF, dwa, dba, pad
int launch_word_table_bwd(const float* SF, const float* DF, const float* wa, const float* dT, int tokens, float* dSF,
                          float* out, float* partial, cudaStream_t st) {
    const int warps = word_table_parts(tokens);
    word_table_bwd_kernel<<<warps / 4, 128, 0, st>>>(SF, DF, wa, dT, tokens, dSF, partial);
    GCGCN_CHECK_LAUNCH("word_table_bwd");
    return launch_reduce_partials(partial, warps, WT_PARTIAL, out, WT_PARTIAL, nullptr, st);
}

static bool word_pool_doc_path(const gcgcn_edge_tables* t) {
    return t->num_active_docs > 0 && t->max_active_len > 0 && t->max_active_len <= WP_MAX_LEN && t->adoc_tok0 != nullptr &&
           t->adoc_len != nullptr && t->adoc_slot_lo != nullptr && t->adoc_slot_hi != nullptr;
}

int launch_word_pool_fwd(const gcgcn_edge_tables* t, const float* T, const float* ctx, float* att, float* cwa,
                         cudaStream_t st) {
    if (t->num_slots <= 0) return GCGCN_OK;
    if (word_pool_doc_path(t)) {
        const size_t smem = static_cast<size_t>(t->max_active_len) * (D + EF_BUCKETS) * sizeof(float);
        GCGCN_TRY(set_smem(word_pool_fwd_doc_kernel, smem, "word_pool_fwd smem"));   // (the size varies with the batch)
        word_pool_fwd_doc_kernel<<<t->num_active_docs, 256, smem, st>>>(make_tabs(t), T, ctx, att, cwa);
        GCGCN_CHECK_LAUNCH("word_pool_fwd<doc>");
        return GCGCN_OK;
    }
    word_pool_fwd_kernel<<<warps_grid(2LL * t->num_slots, 8), 256, 0, st>>>(make_tabs(t), T, ctx, att, cwa);
    GCGCN_CHECK_LAUNCH("word_pool_fwd");
    return GCGCN_OK;
}

int launch_word_pool_bwd(const gcgcn_edge_tables* t, const float* ctx, const float* att, const float* dcwa, float* dlog,
                         float* dctx, float* dT, cudaStream_t st) {
    if (t->num_slots <= 0 || t->num_tokens <= 0) return GCGCN_OK;
    const EdgeTabs tb = make_tabs(t);
    if (word_pool_doc_path(t)) {
        const size_t L = static_cast<size_t>(t->max_active_len);
        const size_t smem = (L * (D + 32) + WP_ENT * D + 2 * WP_ENT * (L + 1)) * sizeof(float);
        GCGCN_TRY(set_smem(word_pool_bwd_doc_kernel, smem, "word_pool_bwd smem"));
        word_pool_bwd_doc_kernel<<<t->num_active_docs, 256, smem, st>>>(tb, ctx, att, dcwa, dctx, dT);
        GCGCN_CHECK_LAUNCH("word_pool_bwd<doc>");
        return GCGCN_OK;
    }
    word_pool_bwd_logit_kernel<<<warps_grid(2LL * t->num_slots, 8), 256, 0, st>>>(tb, ctx, att, dcwa, dlog);
    GCGCN_CHECK_LAUNCH("word_pool_bwd_logit");
    word_pool_bwd_token_kernel<<<warps_grid(t->num_tokens, 8), 256, 0, st>>>(tb, att, dlog, dcwa, dctx, dT);
    GCGCN_CHECK_LAUNCH("word_pool_bwd_token");
    return GCGCN_OK;
}

int launch_sent_pool_fwd(const gcgcn_edge_tables* t, const float* cw, const float* sfeat, const float* nfeat,
                         const float* va, const float* ca, float* score, float* csa, cudaStream_t st) {
    if (t->num_pairs <= 0) return GCGCN_OK;
    sent_pool_fwd_kernel<<<warps_grid(t->num_pairs, 8), 256, 0, st>>>(make_tabs(t), cw, sfeat, nfeat, va, ca, score, csa);
    GCGCN_CHECK_LAUNCH("sent_pool_fwd");
    return GCGCN_OK;
}

int sent_pool_parts(int pairs) { return std::max(1, std::min(sm_count() * 8, (pairs + 3) / 4)) * 4; }

// out: [128 + 4] = dva, dca, pad;  dnfeat: [total_nodes, 128]
int launch_sent_pool_bwd(const gcgcn_edge_tables* t, int total_nodes, const float* cw, const float* sfeat,
                         const float* nfeat, const float* va, const float* score, const float* dcsa, float* dcw,
                         float* dsfeat, float* dnfeat, float* out, float* dpre, float* partial, cudaStream_t st) {
    const int warps = sent_pool_parts(t->num_pairs);
    sent_pool_bwd_kernel<<<warps / 4, 128, 0, st>>>(make_tabs(t), cw, sfeat, nfeat, va, score, dcsa, dcw, dsfeat, dpre,
                                                   partial);
    GCGCN_CHECK_LAUNCH("sent_pool_bwd");
    GCGCN_TRY(launch_reduce_partials(partial, warps, SP_PARTIAL, out, SP_PARTIAL, nullptr, st));
    if (total_nodes > 0) {
        node_collect_kernel<<<warps_grid(total_nodes, 8), 256, 0, st>>>(t->node_ctr_ptr, t->node_ctr, dpre, total_nodes,
                                                                       dnfeat);
        GCGCN_CHECK_LAUNCH("sent_pool_node_collect");
    }
    return GCGCN_OK;
}

template <typename T>
static int edge_fill_t(const float* bias, const float* rows, const long long* pair_idx, int pairs, long long total_pairs,
                       T* e, cudaStream_t st) {
    const long long n4 = total_pairs * (D / 4);
    edge_fill_kernel<T><<<static_cast<unsigned>((n4 + 255) / 256), 256, 0, st>>>(bias, total_pairs, e);
    GCGCN_CHECK_LAUNCH("edge_fill");
    if (pairs > 0) {
        edge_scatter_kernel<T><<<warps_grid(pairs, 8), 256, 0, st>>>(bias, rows, pair_idx, pairs, e);
        GCGCN_CHECK_LAUNCH("edge_fill_scatter");
    }
    return GCGCN_OK;
}

int launch_edge_fill_fwd(const float* bias, const float* rows, const void* pair_idx, int pairs, long long total_pairs,
                         int dtype, void* e, cudaStream_t st) {
    if (total_pairs <= 0) return GCGCN_OK;
    const long long* pi = static_cast<const long long*>(pair_idx);
    if (dtype == GCGCN_F32) return edge_fill_t<float>(bias, rows, pi, pairs, total_pairs, static_cast<float*>(e), st);
    if (dtype == GCGCN_BF16)
        return edge_fill_t<__nv_bfloat16>(bias, rows, pi, pairs, total_pairs, static_cast<__nv_bfloat16*>(e), st);
    return fail(GCGCN_ERR_UNSUPPORTED, "edge dtype %d not supported", dtype);
}

int edge_colsum_parts(long long total_pairs) {
    return static_cast<int>(std::max<long long>(1, std::min<long long>(sm_count() * 8, (total_pairs + 63) / 64)));
}

template <typename T>
static int edge_fill_bwd_t(const T* de, const long long* pair_idx, int pairs, long long total_pairs, float* drows,
                           float* dbias, float* partial, cudaStream_t st) {
    if (pairs > 0) {
        edge_gather_kernel<T><<<warps_grid(pairs, 8), 256, 0, st>>>(de, pair_idx, pairs, drows);
        GCGCN_CHECK_LAUNCH("edge_fill_gather");
    }
    const int parts = edge_colsum_parts(total_pairs);
    const long long rpb = (total_pairs + parts - 1) / parts;
    edge_colsum_kernel<T><<<parts, 256, 0, st>>>(de, total_pairs, rpb, partial);
    GCGCN_CHECK_LAUNCH("edge_fill_colsum");
    return launch_reduce_partials(partial, parts, D, dbias, D, nullptr, st);
}

int launch_edge_fill_bwd(const void* de, const void* pair_idx, int pairs, long long total_pairs, int dtype, float* drows,
                         float* dbias, float* partial, cudaStream_t st) {
    const long long* pi = static_cast<const long long*>(pair_idx);
    if (dtype == GCGCN_F32)
        return edge_fill_bwd_t<float>(static_cast<const float*>(de), pi, pairs, total_pairs, drows, dbias, partial, st);
    if (dtype == GCGCN_BF16)
        return edge_fill_bwd_t<__nv_bfloat16>(static_cast<const __nv_bfloat16*>(de), pi, pairs, total_pairs, drows, dbias,
                                              partial, st);
    return fail(GCGCN_ERR_UNSUPPORTED, "edge dtype %d not supported", dtype);
}

}  // namespace gcgcn
