// extern "C" surface of libgcgcn_b200.so (declared in include/gcgcn_b200.h).
// Host-side orchestration only: argument checks, workspace carving and kernel sequencing.
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"

namespace gcgcn {

// ---- launchers implemented in the kernel files ---------------------------------------------
int launch_node_score(const float* x, const float* u, const float* c, float* ux, int rows, cudaStream_t st);
int launch_edge_fwd(const gcgcn_batch* bt, const void* e, int dtype, const float* v, const float* ux,
                    const uint8_t* mask, const float* keep, float* P, float* A, float* ebar, cudaStream_t st);
int launch_edge_bwd(const gcgcn_batch* bt, const void* e, int dtype, const float* v, const float* dS,
                    const float* debar, void* de, float* dv_partial, cudaStream_t st);
int edge_bwd_grid();
int node_bwd_grid();
int launch_softmax_bwd(const gcgcn_batch* bt, int heads, const float* P, const float* keep, const float* dA,
                       const uint8_t* mask, float* dS, cudaStream_t st);
int launch_gat_node_bwd(const gcgcn_batch* bt, const float* dS, const float* x, const float* u, float* dx,
                        float* partial, int* parts_out, cudaStream_t st);
int launch_reduce_partials(const float* partial, int parts, int width, float* out0, int width0, float* out1,
                           cudaStream_t st);
int launch_mha_fwd(const gcgcn_batch* bt, int heads, const float* q, const float* keep, float* P, float* A,
                   cudaStream_t st);
int launch_mha_bwd(const gcgcn_batch* bt, int heads, const float* q, const float* dS, float* dq, cudaStream_t st);
int launch_stack_fwd(const gcgcn_batch* bt, int heads, int layers, int slab, int flags, const float* A, float* Z,
                     const float* E, const float* Winner, const float* keep, const float* x, float* G, float* F,
                     float* frag_ws, cudaStream_t st);
int launch_stack_bwd(const gcgcn_batch* bt, int heads, int layers, int slab, int flags, const float* A, const float* Z,
                     const float* G, const float* Winner, const float* keep, const float* dF, float* dZ,
                     float* dE, float* dA, float* frag_ws, cudaStream_t st);
bool block_kernels_usable(const gcgcn_batch* bt, int heads, int layers, int slab, bool mha);
bool set_tile_blocks(bool on);
int launch_block_fwd(const gcgcn_batch* bt, int heads, int layers, const float* A, const float* q, float* P,
                     float* Z, const float* E, const float* Winner, const float* x, float* G, float* F,
                     float* frag_ws, const BlockDrop& drop, cudaStream_t st);
int launch_block_bwd(const gcgcn_batch* bt, int heads, int layers, int out_mode, const float* A, const float* q,
                     const float* Z, const float* G, const float* Winner, const float* dF, float* dZ, float* dE,
                     float* dOut, float* frag_ws, const BlockDrop& drop, cudaStream_t st);
int launch_dropout_mask(unsigned long long seed, uint32_t stream, uint32_t thr, float inv, long long count, float* out,
                        cudaStream_t st);
size_t block_frag_floats(int heads, int layers);
enum { ATT_GRAD_DA = 0, ATT_GRAD_DS = 1, ATT_GRAD_DQ = 2 };   // == BK_OUT_* of gcn_block.cu
int launch_gemm(int ta, int tb, int M, int N, int K, float alpha, const float* A, int lda, const float* B,
                int ldb, float beta, float* C, int ldc, const float* bias, void* ws, size_t ws_bytes,
                cudaStream_t st);
size_t gemm_presplit_bytes(int rows);
int launch_colsum(const float* X, int M, int N, int ldx, float* out, void* ws, size_t ws_bytes, cudaStream_t st);
int launch_gemm_batched(int ta, int tb, int M, int N, int K, float alpha, const float* A, int lda, const float* B,
                        int ldb, float beta, float* C, int ldc, int batch, long long sA, long long sB, long long sC,
                        void* ws, size_t ws_bytes, cudaStream_t st);
int launch_csr_gather(const float* src, const int* ptr, const int* idx, const float* w, int rows, float* out,
                      cudaStream_t st);
int launch_pair_gather_fwd(const gcgcn_batch* bt, const float* feat, int feat_w, const float* dis, int dis_w,
                           const int* h_idx, const int* t_idx, const int* dis_h, const int* dis_t, float* out_h,
                           float* out_t, cudaStream_t st);
int launch_pair_gather_bwd(const gcgcn_batch* bt, const float* dout_h, const float* dout_t, int feat_w,
                           int dis_w, int dis_rows, const int* dis_h, const int* dis_t, float* dfeat,
                           float* ddis, void* ws, size_t ws_bytes, cudaStream_t st);
int pair_dis_warps();
int launch_pair_dense_fwd(const gcgcn_batch* bt, const float* U, const float* Vd, const int* h_idx, const int* t_idx,
                          const int* dis_h, const int* dis_t, float* out_h, float* out_t, cudaStream_t st);
int launch_pair_dense_bwd(const gcgcn_batch* bt, const float* dout_h, const float* dout_t, const float* out_h,
                          const float* out_t, int dis_rows, const int* dis_h, const int* dis_t, float* dU, float* dVd,
                          float* dpre, void* ws, size_t ws_bytes, cudaStream_t st);
int launch_pack_stack(const float* const* wn_ptrs, const float* const* we_ptrs, int heads, int layers, int slab,
                      float* WnX, float* We, float* Winner, cudaStream_t st);
int launch_expand_pair_context(const int* slots, int num_slots, int n, int S, int L, int dis_plus, unsigned char* sen,
                               long long* pos_h, long long* pos_t, cudaStream_t st);
int launch_adam(float* p, const float* g, float* m, float* v, long long count, float lr, float b1, float b2,
                float eps, float wd, float gscale, int step, cudaStream_t st);
int launch_unpack_stack(const float* dWnX, const float* dWe, const float* dWinner, int heads, int layers, int slab,
                        float* dwn_flat, float* dwe_flat, cudaStream_t st);

int launch_word_table_fwd(const float* SF, const float* DF, const float* wa, const float* ba, int tokens, float* T,
                          cudaStream_t st);
int word_table_parts(int tokens);
int launch_word_table_bwd(const float* SF, const float* DF, const float* wa, const float* dT, int tokens, float* dSF,
                          float* out, float* partial, cudaStream_t st);
int launch_word_pool_fwd(const gcgcn_edge_tables* t, const float* T, const float* ctx, float* att, float* cwa,
                         cudaStream_t st);
int launch_word_pool_bwd(const gcgcn_edge_tables* t, const float* ctx, const float* att, const float* dcwa, float* dlog,
                         float* dctx, float* dT, cudaStream_t st);
int launch_sent_pool_fwd(const gcgcn_edge_tables* t, const float* cw, const float* sfeat, const float* nfeat,
                         const float* va, const float* ca, float* score, float* csa, cudaStream_t st);
int sent_pool_parts(int pairs);
int launch_sent_pool_bwd(const gcgcn_edge_tables* t, int total_nodes, const float* cw, const float* sfeat,
                         const float* nfeat, const float* va, const float* score, const float* dcsa, float* dcw,
                         float* dsfeat, float* dnfeat, float* out, float* dpre, float* partial, cudaStream_t st);
int launch_edge_fill_fwd(const float* bias, const float* rows, const void* pair_idx, int pairs, long long total_pairs,
                         int dtype, void* e, cudaStream_t st);
int edge_colsum_parts(long long total_pairs);
int launch_edge_fill_bwd(const void* de, const void* pair_idx, int pairs, long long total_pairs, int dtype, float* drows,
                         float* dbias, float* partial, cudaStream_t st);

int launch_bilinear_reduce(const float* Y, const float* t, const float* bias, int rows, int R, int accumulate, float* out,
                           int ldo, cudaStream_t st);
int launch_bilinear_finish(const float* part, long long ld, const float* bias, int rows, int R, int accumulate, float* out,
                           int ldo, cudaStream_t st);
int launch_gemm_rowop(int mode, int M, int N, int K, const float* A, int lda, const float* B, int ldb, const float* T,
                      float* out, long long ld, void* ws, size_t ws_bytes, cudaStream_t st);
int launch_gemm_wgrad_scaled(int M, int tiles, int K, const float* A, int lda, const float* T, const float* scale, int lds,
                             float beta, float* C, int ldc, void* ws, size_t ws_bytes, cudaStream_t st, void* pre_ws,
                             size_t pre_bytes);
int launch_bilinear_outer(const float* dout, int ldd, const float* t, int rows, int R, float* dY, cudaStream_t st);
int launch_bilinear_dt(const float* dout, int ldd, const float* Y, int rows, int R, float* dt, cudaStream_t st);
int launch_doc_bias_fwd(const gcgcn_batch* bt, const float* v, int R, float* z, cudaStream_t st);
int launch_doc_bias_bwd(const gcgcn_batch* bt, const float* dz, int R, float* dv, cudaStream_t st);
int launch_pair_bce_fwd(const gcgcn_batch* bt, const float* z, const float* y, int R, float* loss, cudaStream_t st);
int launch_pair_bce_bwd(const gcgcn_batch* bt, const float* z, const float* y, int R, const float* dloss, float* dz,
                        cudaStream_t st);

int launch_gat_collapse_fwd(const float* Wh, const float* bh, const float* Wt, const float* bt, const float* Wr,
                            const float* br, const float* w, const float* b, int hid, float* out, cudaStream_t st);
int launch_gat_collapse_bwd(const float* Wh, const float* bh, const float* Wt, const float* bt, const float* Wr,
                            const float* br, const float* w, const float* dout, int hid, float* dWh, float* dbh, float* dWt,
                            float* dbt, float* dWr, float* dbr, float* dw, float* db, cudaStream_t st);
int launch_pack_rows(const float* const* ptrs, int count, int elems, float* out, cudaStream_t st);
size_t rank_ws_bytes(long long count);
int launch_rank_candidates(const gcgcn_batch* bt, const float* z, const float* labels, const uint8_t* intrain, int R,
                           long long base_id, float* score, uint32_t* payload, unsigned long long* counters,
                           cudaStream_t st);
int launch_rank_sort(const float* score, const uint32_t* payload, long long count, uint32_t* sorted_key,
                     uint32_t* sorted_payload, void* ws, size_t ws_bytes, cudaStream_t st);
int launch_rank_curve(const uint32_t* key, const uint32_t* pay, long long count, long long T, int has_intrain,
                      double input_theta, gcgcn_rank_result* res, void* ws, size_t ws_bytes, cudaStream_t st);
int launch_rank_candidates_at(const gcgcn_batch* bt, const float* z, const float* labels, const uint8_t* intrain,
                              int R, const long long* doc_first, float* score, uint32_t* payload,
                              unsigned long long* counters, cudaStream_t st);
size_t rank_merge_ws_bytes(long long count);
int launch_rank_merge(const uint32_t* key_a, const uint32_t* pay_a, long long na, const uint32_t* key_b,
                      const uint32_t* pay_b, long long nb, uint32_t* key_out, uint32_t* pay_out, void* ws,
                      size_t ws_bytes, cudaStream_t st);
int launch_rank_curve_points(const uint32_t* pay, long long count, long long T, int has_intrain, float* x, float* y,
                             float* yi, void* ws, size_t ws_bytes, cudaStream_t st);
size_t rank_relations_ws_bytes(long long count, int R);
int launch_rank_by_relation(const uint32_t* key, const uint32_t* pay, long long count, int R, uint32_t* rel_key,
                            uint32_t* rel_pay, void* ws, size_t ws_bytes, cudaStream_t st);
int launch_rank_curve_relations(const uint32_t* key, const uint32_t* pay, long long count, int R,
                                const long long* total_recall, int has_intrain, const double* input_theta,
                                gcgcn_rank_result* res, void* ws, size_t ws_bytes, cudaStream_t st);
int launch_rank_select(const uint32_t* key, const uint32_t* pay, long long count, int R, const float* theta,
                       uint32_t* out_key, uint32_t* out_pay, long long* counts, void* ws, size_t ws_bytes,
                       cudaStream_t st);
int launch_rank_decode(const uint32_t* key, const uint32_t* pay, long long rows, const long long* doc_off,
                       const int* doc_n, int docs, int R, int* doc, int* row, int* col, int* rel, float* score,
                       cudaStream_t st);

// ---- error text, launch counter, device cache --------------------------------------------------
std::atomic<uint64_t> g_launches{0};
std::atomic<bool> g_timing{false};

namespace {
struct Mark { const char* name; cudaEvent_t ev; cudaStream_t st; double work; };
thread_local double g_pending_work = 0.0;
std::mutex g_tmutex;
std::vector<Mark> g_marks;
std::vector<cudaEvent_t> g_event_pool;
cudaEvent_t take_event() {
    if (!g_event_pool.empty()) { cudaEvent_t e = g_event_pool.back(); g_event_pool.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}
}  // namespace

void timing_mark(const char* name, cudaStream_t st) {
    std::lock_guard<std::mutex> lk(g_tmutex);
    cudaEvent_t e = take_event();
    if (e == nullptr) return;
    cudaEventRecord(e, st);
    g_marks.push_back({name, e, st, g_pending_work});
    g_pending_work = 0.0;
}

void timing_set_work(double work) {
    if (g_timing.load(std::memory_order_relaxed)) g_pending_work = work;
}

char* error_buffer() {
    static thread_local char buf[512] = "";
    return buf;
}

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(error_buffer(), 512, fmt, ap);
    va_end(ap);
    return code;
}

int sm_count() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

int check_device_ptr(const void* p, const char* name) {
    if (p == nullptr) return fail(GCGCN_ERR_INVALID_ARG, "%s is NULL", name);
    cudaPointerAttributes attr;
    cudaError_t e = cudaPointerGetAttributes(&attr, p);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(GCGCN_ERR_INVALID_ARG, "%s: not a CUDA pointer (%s); this library has no CPU path", name,
                    cudaGetErrorString(e));
    }
    if (attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged)
        return fail(GCGCN_ERR_INVALID_ARG, "%s is host memory; this library has no CPU path", name);
    return GCGCN_OK;
}

int check_batch(const gcgcn_batch* bt) {
    if (bt == nullptr) return fail(GCGCN_ERR_INVALID_ARG, "batch descriptor is NULL");
    if (bt->num_docs < 0 || bt->total_nodes < 0 || bt->total_pairs < 0 || bt->max_nodes < 0)
        return fail(GCGCN_ERR_INVALID_ARG, "negative size in batch descriptor");
    if (bt->num_docs > 0) {
        GCGCN_TRY(check_device_ptr(bt->node_ptr, "batch.node_ptr"));
        GCGCN_TRY(check_device_ptr(bt->pair_ptr, "batch.pair_ptr"));
        GCGCN_TRY(check_device_ptr(bt->row_doc, "batch.row_doc"));
    }
    return GCGCN_OK;
}

constexpr size_t GEMM_WS_BYTES = size_t(24) << 20;
constexpr int BLOCK_FLAGS_ALL = GCGCN_STACK_RELU | GCGCN_STACK_RESIDUAL | GCGCN_STACK_LINEAR;

static size_t align256(size_t b) { return (b + 255) & ~size_t(255); }

// dropout streams of the two blocks (distinct masks for distinct tensors under one seed)
enum { DROP_STREAM_GAT = 1, DROP_STREAM_CAGGC = 2, DROP_STREAM_MHA = 3, DROP_STREAM_MAGGC = 4 };

static uint32_t drop_threshold(float p) {
    if (!(p > 0.f)) return 0u;
    const double t = static_cast<double>(p) * 4294967296.0;
    return t >= 4294967295.0 ? 4294967295u : static_cast<uint32_t>(t);
}
static int make_block_drop(const gcgcn_dropout* d, uint32_t s_att, uint32_t s_gcn, BlockDrop* out) {
    *out = BlockDrop{};
    if (d == nullptr) return GCGCN_OK;
    if (!(d->p_att >= 0.f && d->p_att < 1.f && d->p_gcn >= 0.f && d->p_gcn < 1.f))
        return fail(GCGCN_ERR_INVALID_ARG, "dropout probabilities must be in [0, 1): p_att %g, p_gcn %g", d->p_att, d->p_gcn);
    out->seed = d->seed;
    out->thr_att = drop_threshold(d->p_att);
    out->thr_gcn = drop_threshold(d->p_gcn);
    out->inv_att = 1.0f / (1.0f - d->p_att);
    out->inv_gcn = 1.0f / (1.0f - d->p_gcn);
    out->s_att = s_att;
    out->s_gcn = s_gcn;
    return GCGCN_OK;
}
static bool drop_active(const BlockDrop& d) { return d.thr_att != 0u || d.thr_gcn != 0u; }

__global__ void __launch_bounds__(256)
head_sum_kernel(const float* __restrict__ dF, int heads, int rows, float* __restrict__ dx) {
    const size_t idx = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;  // float4 index
    if (idx >= static_cast<size_t>(rows) * (D / 4)) return;
    const size_t r = idx / (D / 4), q = idx % (D / 4);
    const float4* src = reinterpret_cast<const float4*>(dF) + r * heads * (D / 4) + q;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int h = 0; h < heads; ++h) {
        const float4 v = src[static_cast<size_t>(h) * (D / 4)];
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    reinterpret_cast<float4*>(dx)[idx] = acc;
}

__global__ void __launch_bounds__(256) add_kernel(float* __restrict__ dst, const float* __restrict__ src, size_t n4) {
    const size_t idx = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= n4) return;
    float4 a = reinterpret_cast<float4*>(dst)[idx];
    const float4 b = reinterpret_cast<const float4*>(src)[idx];
    a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    reinterpret_cast<float4*>(dst)[idx] = a;
}

// dst += src, n a multiple of 4
static int launch_add(float* dst, const float* src, size_t n, cudaStream_t st) {
    if (n == 0) return GCGCN_OK;
    add_kernel<<<ceil_div(n / 4, 256), 256, 0, st>>>(dst, src, n / 4);
    GCGCN_CHECK_LAUNCH("add");
    return GCGCN_OK;
}

// Wsum[d][c] = sum_h Wout[d][h * 128 + c]: with dF = dy Wout, the residual's share sum_h dF_h of dx is dy Wsum -- a
// [rows, 128] x [128, 128] product instead of a pass over the [rows, heads * 128] slab
__global__ void __launch_bounds__(256)
wout_head_sum_kernel(const float* __restrict__ Wout, int heads, float* __restrict__ Wsum) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;       // over D * D
    if (idx >= D * D) return;
    const int d = idx / D, c = idx - d * D;
    float acc = 0.f;
    for (int h = 0; h < heads; ++h) acc += Wout[static_cast<size_t>(d) * heads * D + h * D + c];
    Wsum[idx] = acc;
}

static int launch_head_sum(const float* dF, int heads, int rows, float* dx, cudaStream_t st) {
    if (rows == 0) return GCGCN_OK;
    const size_t total = static_cast<size_t>(rows) * (D / 4);
    head_sum_kernel<<<ceil_div(total, 256), 256, 0, st>>>(dF, heads, rows, dx);
    GCGCN_CHECK_LAUNCH("head_sum");
    return GCGCN_OK;
}

}  // namespace gcgcn

using namespace gcgcn;

extern "C" {

const char* gcgcn_version(void) { return "gcgcn_b200 0.1.0 (sm_100a)"; }
const char* gcgcn_last_error(void) { return error_buffer(); }
uint64_t gcgcn_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
int32_t gcgcn_set_tile_blocks(int32_t enable) { return gcgcn::set_tile_blocks(enable != 0) ? 1 : 0; }

int gcgcn_device_info(int32_t* sms, int32_t* major, int32_t* minor) {
    int dev = 0;
    GCGCN_TRY(cuda_ok(cudaGetDevice(&dev), "cudaGetDevice"));
    int a = 0, b = 0, c = 0;
    GCGCN_TRY(cuda_ok(cudaDeviceGetAttribute(&a, cudaDevAttrMultiProcessorCount, dev), "device attr"));
    GCGCN_TRY(cuda_ok(cudaDeviceGetAttribute(&b, cudaDevAttrComputeCapabilityMajor, dev), "device attr"));
    GCGCN_TRY(cuda_ok(cudaDeviceGetAttribute(&c, cudaDevAttrComputeCapabilityMinor, dev), "device attr"));
    if (sms) *sms = a;
    if (major) *major = b;
    if (minor) *minor = c;
    return GCGCN_OK;
}

size_t gcgcn_workspace_bytes(int32_t total_nodes, int64_t total_pairs, int32_t heads) {
    const size_t hd = static_cast<size_t>(heads < 1 ? 1 : heads) * D;
    const size_t nodes = static_cast<size_t>(total_nodes < 0 ? 0 : total_nodes);
    const size_t pairs = static_cast<size_t>(total_pairs < 0 ? 0 : total_pairs);
    size_t b = 0;
    b += 3 * align256(nodes * hd * sizeof(float));                     // dF, dZ, dE
    b += align256(pairs * (heads < 1 ? 1 : heads) * sizeof(float));    // dS
    b += 2 * align256(nodes * D * sizeof(float));                      // dq / ux / misc
    b += GEMM_WS_BYTES + (size_t(8) << 20);                            // split-K and reduction partials
    b += size_t(4) << 20;                                              // fragment-ordered dense-connect weights
    b += size_t(256) << 10;                                            // head-summed output weights
    return b;
}

// ---- per-kernel timing (bench.py's roofline section) ----------------------------------------
int gcgcn_timing_begin(void* stream) {
    std::lock_guard<std::mutex> lk(g_tmutex);
    for (auto& m : g_marks) g_event_pool.push_back(m.ev);
    g_marks.clear();
    cudaEvent_t e = take_event();
    if (e == nullptr) return fail(GCGCN_ERR_CUDA, "timing_begin: cannot create an event");
    GCGCN_TRY(cuda_ok(cudaEventRecord(e, static_cast<cudaStream_t>(stream)), "timing_begin"));
    g_marks.push_back({"(begin)", e, static_cast<cudaStream_t>(stream), 0.0});
    g_timing.store(true);
    return GCGCN_OK;
}

// writes one line per kernel name: "<name>\t<launches>\t<total milliseconds>\t<total work (flop)>\n"
int gcgcn_timing_end(void* stream, char* buf, size_t cap) {
    g_timing.store(false);
    std::lock_guard<std::mutex> lk(g_tmutex);
    (void)stream;
    if (buf == nullptr || cap == 0) return fail(GCGCN_ERR_INVALID_ARG, "timing_end: no buffer");
    buf[0] = 0;
    if (g_marks.empty()) return GCGCN_OK;
    GCGCN_TRY(cuda_ok(cudaEventSynchronize(g_marks.back().ev), "timing_end"));
    GCGCN_TRY(cuda_ok(cudaDeviceSynchronize(), "timing_end"));
    struct Acc { long count = 0; double ms = 0.0, work = 0.0; };
    std::map<std::string, Acc> acc;
    std::map<cudaStream_t, cudaEvent_t> last;          // a kernel's time = gap to the previous mark on ITS stream
    for (size_t i = 0; i < g_marks.size(); ++i) {
        auto it = last.find(g_marks[i].st);
        if (it != last.end()) {
            float ms = 0.f;
            // host-side gaps are only meaningful on the stream timing_begin was called on
            const bool gap_mark = g_marks[i].name[0] == '(';
            if (gap_mark && g_marks[i].st != g_marks[0].st) {
                // chain reset only
            } else if (cudaEventElapsedTime(&ms, it->second, g_marks[i].ev) == cudaSuccess) {
                auto& slot = acc[g_marks[i].name];
                slot.count += 1;
                slot.ms += ms;
                slot.work += g_marks[i].work;
            } else {
                cudaGetLastError();
            }
        }
        last[g_marks[i].st] = g_marks[i].ev;
    }
    size_t off = 0;
    for (auto& kv : acc) {
        int w = snprintf(buf + off, cap - off, "%s\t%ld\t%.6f\t%.6e\n", kv.first.c_str(), kv.second.count, kv.second.ms,
                         kv.second.work);
        if (w < 0 || static_cast<size_t>(w) >= cap - off) break;
        off += static_cast<size_t>(w);
    }
    for (auto& m : g_marks) g_event_pool.push_back(m.ev);
    g_marks.clear();
    return GCGCN_OK;
}

// ---- a1 pooling ------------------------------------------------------------------------------
int gcgcn_pool_fwd(const float* ctx, const int32_t* ent_ptr, const int32_t* tok_idx, const float* w,
                   int32_t total_nodes, float* x0, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(total_nodes >= 0, "pool_fwd: total_nodes < 0");
    if (total_nodes == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(ctx, "ctx"));
    GCGCN_TRY(check_device_ptr(ent_ptr, "ent_ptr"));
    GCGCN_TRY(check_device_ptr(x0, "x0"));
    return launch_csr_gather(ctx, ent_ptr, tok_idx, w, total_nodes, x0, static_cast<cudaStream_t>(stream));
}

int gcgcn_pool_bwd(const float* dx0, const int32_t* tok_ptr, const int32_t* ent_idx, const float* w_t,
                   int32_t total_tokens, float* dctx, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(total_tokens >= 0, "pool_bwd: total_tokens < 0");
    if (total_tokens == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(dx0, "dx0"));
    GCGCN_TRY(check_device_ptr(tok_ptr, "tok_ptr"));
    GCGCN_TRY(check_device_ptr(dctx, "dctx"));
    return launch_csr_gather(dx0, tok_ptr, ent_idx, w_t, total_tokens, dctx, static_cast<cudaStream_t>(stream));
}

// ---- shared edge pass ------------------------------------------------------------------------
int gcgcn_edge_mean_fwd(const gcgcn_batch* bt, const void* e, int32_t edge_dtype, float* ebar, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_batch(bt));
    if (bt->total_nodes == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(e, "edge_feat"));
    GCGCN_TRY(check_device_ptr(ebar, "ebar"));
    return launch_edge_fwd(bt, e, edge_dtype, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, ebar,
                           static_cast<cudaStream_t>(stream));
}

int gcgcn_edge_mean_bwd(const gcgcn_batch* bt, const float* debar, int32_t edge_dtype, void* de, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_batch(bt));
    if (bt->total_nodes == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(debar, "debar"));
    GCGCN_TRY(check_device_ptr(de, "de"));
    return launch_edge_bwd(bt, nullptr, edge_dtype, nullptr, nullptr, debar, de, nullptr,
                           static_cast<cudaStream_t>(stream));
}

// ---- a2 GATAttention -------------------------------------------------------------------------
int gcgcn_gat_fwd(const gcgcn_batch* bt, const float* x, const void* e, int32_t edge_dtype, const float* u,
                  const float* v, const float* c, const uint8_t* mask, int32_t apply_mask, const float* keep,
                  float* P, float* A, float* ebar, void* ws, size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_batch(bt));
    if (bt->total_nodes == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(x, "node_feat"));
    GCGCN_TRY(check_device_ptr(e, "edge_feat"));
    GCGCN_TRY(check_device_ptr(u, "u"));
    GCGCN_TRY(check_device_ptr(v, "v"));
    GCGCN_TRY(check_device_ptr(P, "P"));
    GCGCN_TRY(check_device_ptr(A, "A"));
    GCGCN_TRY(check_device_ptr(ebar, "ebar"));
    GCGCN_REQUIRE(keep == nullptr || A != P, "gat_fwd: A must not alias P when a keep mask is given");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    Arena ar(ws, ws_bytes);
    float* ux = ar.take<float>(bt->total_nodes);
    if (ux == nullptr) return fail(GCGCN_ERR_WORKSPACE, "gat_fwd: workspace too small");
    GCGCN_TRY(launch_node_score(x, u, c, ux, bt->total_nodes, st));
    return launch_edge_fwd(bt, e, edge_dtype, v, ux, (apply_mask ? mask : nullptr), keep, P, A, ebar, st);
}

// GAT backward downstream of the softmax: dS -> dx (node half), du, dc, and the edge pass (de, dv).
static int gat_bwd_from_ds(const gcgcn_batch* bt, const float* x, const void* e, int32_t edge_dtype, const float* u,
                           const float* v, const float* dS, const float* debar, float* dx, void* de, float* du,
                           float* dv, float* dc, Arena& ar, cudaStream_t st) {
    float* node_part = ar.take<float>(static_cast<size_t>(node_bwd_grid()) * (D + 1));
    float* dv_part = ar.take<float>(static_cast<size_t>(edge_bwd_grid()) * D);
    if (node_part == nullptr || dv_part == nullptr) return fail(GCGCN_ERR_WORKSPACE, "gat_bwd: workspace too small");
    int parts = 0;
    GCGCN_TRY(launch_gat_node_bwd(bt, dS, x, u, dx, node_part, &parts, st));
    GCGCN_TRY(launch_reduce_partials(node_part, parts, D + 1, du, D, dc, st));
    GCGCN_TRY(launch_edge_bwd(bt, e, edge_dtype, v, dS, debar, de, dv_part, st));
    const int grid = edge_bwd_grid() < bt->total_nodes ? edge_bwd_grid() : bt->total_nodes;
    return launch_reduce_partials(dv_part, grid, D, dv, D, nullptr, st);
}

int gcgcn_gat_bwd(const gcgcn_batch* bt, const float* x, const void* e, int32_t edge_dtype, const float* u,
                  const float* v, const uint8_t* mask, int32_t apply_mask, const float* keep, const float* P,
                  const float* dA, const float* debar, float* dx, void* de, float* du, float* dv, float* dc,
                  void* ws, size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_batch(bt));
    if (bt->total_nodes == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(x, "node_feat"));
    GCGCN_TRY(check_device_ptr(e, "edge_feat"));
    GCGCN_TRY(check_device_ptr(P, "P"));
    GCGCN_TRY(check_device_ptr(dA, "dA"));
    GCGCN_TRY(check_device_ptr(dx, "dx"));
    GCGCN_TRY(check_device_ptr(de, "de"));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    Arena ar(ws, ws_bytes);
    float* dS = ar.take<float>(bt->total_pairs);
    if (dS == nullptr) return fail(GCGCN_ERR_WORKSPACE, "gat_bwd: workspace too small");
    GCGCN_TRY(launch_softmax_bwd(bt, 1, P, keep, dA, (apply_mask ? mask : nullptr), dS, st));
    return gat_bwd_from_ds(bt, x, e, edge_dtype, u, v, dS, debar, dx, de, du, dv, dc, ar, st);
}

// ---- a5 MultiHeadAttention -------------------------------------------------------------------
int gcgcn_mha_fwd(const gcgcn_batch* bt, int32_t heads, const float* x, const float* Wq, const float* bq,
                  const float* keep, float* q, float* P, float* A, void* ws, size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_batch(bt));
    GCGCN_REQUIRE(heads >= 1 && D % heads == 0, "mha_fwd: head_num %d must divide %d", heads, D);
    if (bt->total_nodes == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(x, "node_feat"));
    GCGCN_TRY(check_device_ptr(Wq, "Wq"));
    GCGCN_TRY(check_device_ptr(q, "q"));
    GCGCN_TRY(check_device_ptr(P, "P"));
    GCGCN_TRY(check_device_ptr(A, "A"));
    GCGCN_REQUIRE(keep == nullptr || A != P, "mha_fwd: A must not alias P when a keep mask is given");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    GCGCN_TRY(launch_gemm(0, 1, bt->total_nodes, D, D, 1.f, x, D, Wq, D, 0.f, q, D, bq, ws, ws_bytes, st));
    return launch_mha_fwd(bt, heads, q, keep, P, A, st);
}

int gcgcn_mha_bwd(const gcgcn_batch* bt, int32_t heads, const float* x, const float* Wq, const float* q,
                  const float* keep, const float* P, const float* dA, float* dx, float* dWq, float* dbq,
                  void* ws, size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_batch(bt));
    GCGCN_REQUIRE(heads >= 1 && D % heads == 0, "mha_bwd: head_num %d must divide %d", heads, D);
    if (bt->total_nodes == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(x, "node_feat"));
    GCGCN_TRY(check_device_ptr(q, "q"));
    GCGCN_TRY(check_device_ptr(P, "P"));
    GCGCN_TRY(check_device_ptr(dA, "dA"));
    GCGCN_TRY(check_device_ptr(dx, "dx"));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    Arena ar(ws, ws_bytes);
    float* dS = ar.take<float>(static_cast<size_t>(bt->total_pairs) * heads);
    float* dq = ar.take<float>(static_cast<size_t>(bt->total_nodes) * D);
    float* gws = ar.take<float>(GEMM_WS_BYTES / sizeof(float));
    if (dS == nullptr || dq == nullptr || gws == nullptr)
        return fail(GCGCN_ERR_WORKSPACE, "mha_bwd: workspace too small");
    GCGCN_TRY(launch_softmax_bwd(bt, heads, P, keep, dA, nullptr, dS, st));
    GCGCN_TRY(launch_mha_bwd(bt, heads, q, dS, dq, st));
    GCGCN_TRY(launch_gemm(0, 0, bt->total_nodes, D, D, 1.f, dq, D, Wq, D, 0.f, dx, D, nullptr, gws, GEMM_WS_BYTES, st));
    if (dWq != nullptr)
        GCGCN_TRY(launch_gemm(1, 0, D, D, bt->total_nodes, 1.f, dq, D, x, D, 0.f, dWq, D, nullptr, gws, GEMM_WS_BYTES, st));
    if (dbq != nullptr) GCGCN_TRY(launch_colsum(dq, bt->total_nodes, D, D, dbq, gws, GEMM_WS_BYTES, st));
    return GCGCN_OK;
}

// ---- a3/a4/a6 GraphConv stack ----------------------------------------------------------------
// q != nullptr: the attention is the MHA map of q's head slices, computed inside the block kernel (P is written).
static int stack_fwd_impl(const gcgcn_batch* bt, int32_t heads, int32_t layers, int32_t in_dim, int32_t slab,
                          int32_t flags, const float* x, const float* ebar, const float* A, const float* q, float* P,
                          const float* WnX, const float* We, const float* Winner, const float* Wout,
                          const float* bout, const float* keep, float* Z, float* G, float* F, float* y, void* ws,
                          size_t ws_bytes, cudaStream_t st, const BlockDrop& drop = BlockDrop{}) {
    const bool linear = flags & GCGCN_STACK_LINEAR;
    const int HD = heads * slab, M = bt->total_nodes;
    Arena ar(ws, ws_bytes);
    float* E = ar.take<float>(static_cast<size_t>(M) * HD);
    float* gws = ar.take<float>(GEMM_WS_BYTES / sizeof(float));
    float* frag = (slab == D && layers > 1 && D % layers == 0) ? ar.take<float>(block_frag_floats(heads, layers)) : nullptr;
    if (E == nullptr || gws == nullptr) return fail(GCGCN_ERR_WORKSPACE, "stack_fwd: workspace too small");
    GCGCN_TRY(launch_gemm(0, 0, M, HD, in_dim, 1.f, x, in_dim, WnX, HD, 0.f, Z, HD, nullptr, gws, GEMM_WS_BYTES, st));
    GCGCN_TRY(launch_gemm(0, 0, M, HD, D, 1.f, ebar, D, We, HD, 0.f, E, HD, nullptr, gws, GEMM_WS_BYTES, st));
    float* Fout = linear ? F : y;
    if (q != nullptr)
        GCGCN_TRY(launch_block_fwd(bt, heads, layers, nullptr, q, P, Z, E, Winner, x, G, Fout, frag, drop, st));
    else if (drop_active(drop))       // in-kernel dropout exists only in the block kernels (given attention map)
        GCGCN_TRY(launch_block_fwd(bt, heads, layers, A, nullptr, nullptr, Z, E, Winner, x, G, Fout, frag, drop, st));
    else
        GCGCN_TRY(launch_stack_fwd(bt, heads, layers, slab, flags, A, Z, E, Winner, keep, x, G, Fout, frag, st));
    if (linear)
        GCGCN_TRY(launch_gemm(0, 1, M, D, HD, 1.f, F, HD, Wout, HD, 0.f, y, D, bout, gws, GEMM_WS_BYTES, st));
    return GCGCN_OK;
}

int gcgcn_graphconv_stack_fwd(const gcgcn_batch* bt, int32_t heads, int32_t layers, int32_t in_dim,
                              int32_t slab, int32_t flags, const float* x, const float* ebar, const float* A,
                              const float* WnX, const float* We, const float* Winner, const float* Wout,
                              const float* bout, const float* keep, float* Z, float* G, float* F, float* y,
                              void* ws, size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_batch(bt));
    GCGCN_REQUIRE(heads >= 1 && layers >= 1 && in_dim >= 1 && slab >= 1, "stack_fwd: bad heads/layers/widths");
    const bool linear = flags & GCGCN_STACK_LINEAR;
    GCGCN_REQUIRE(linear || heads == 1, "stack_fwd: without the output linear there can be only one head");
    GCGCN_REQUIRE(!(flags & GCGCN_STACK_RESIDUAL) || in_dim == slab,
                  "stack_fwd: the residual needs input width %d == output width %d", in_dim, slab);
    if (bt->total_nodes == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(x, "node_feat"));
    GCGCN_TRY(check_device_ptr(ebar, "ebar"));
    GCGCN_TRY(check_device_ptr(A, "adj_matrix"));
    GCGCN_TRY(check_device_ptr(WnX, "WnX"));
    GCGCN_TRY(check_device_ptr(We, "We"));
    GCGCN_TRY(check_device_ptr(Z, "Z"));
    GCGCN_TRY(check_device_ptr(G, "G"));
    GCGCN_TRY(check_device_ptr(y, "y"));
    if (linear) GCGCN_TRY(check_device_ptr(F, "F"));
    return stack_fwd_impl(bt, heads, layers, in_dim, slab, flags, x, ebar, A, nullptr, nullptr, WnX, We, Winner, Wout,
                          bout, keep, Z, G, F, y, ws, ws_bytes, static_cast<cudaStream_t>(stream));
}

// att_grad: ATT_GRAD_DA -> att_out = dA (any configuration; the caller runs the softmax backward);
//           ATT_GRAD_DS -> att_out = dS (block kernels, one head, A a softmax output);
//           ATT_GRAD_DQ -> att_out = dq [rows][128] (block kernels, A = MHA probabilities of q).
static int stack_bwd_impl(const gcgcn_batch* bt, int32_t heads, int32_t layers, int32_t in_dim, int32_t slab,
                          int32_t flags, int att_grad, const float* x, const float* ebar, const float* A,
                          const float* q, const float* WnX, const float* We, const float* Winner, const float* Wout,
                          const float* keep, const float* Z, const float* G, const float* F, const float* dy,
                          float* dx, float* debar, float* att_out, float* dWnX, float* dWe, float* dWinner,
                          float* dWout, float* dbout, void* ws, size_t ws_bytes, cudaStream_t st,
                          const BlockDrop& drop = BlockDrop{}) {
    const bool linear = flags & GCGCN_STACK_LINEAR;
    const int HD = heads * slab, M = bt->total_nodes, gd = slab / layers;
    Arena ar(ws, ws_bytes);
    float* dFbuf = linear ? ar.take<float>(static_cast<size_t>(M) * HD) : nullptr;
    float* dZ = ar.take<float>(static_cast<size_t>(M) * HD);
    float* dE = ar.take<float>(static_cast<size_t>(M) * HD);
    float* gws = ar.take<float>(GEMM_WS_BYTES / sizeof(float));
    float* frag = (slab == D && layers > 1 && D % layers == 0) ? ar.take<float>(block_frag_floats(heads, layers)) : nullptr;
    if ((linear && dFbuf == nullptr) || dZ == nullptr || dE == nullptr || gws == nullptr)
        return fail(GCGCN_ERR_WORKSPACE, "stack_bwd: workspace too small");
    const float* dF = dy;
    if (linear) {
        GCGCN_TRY(launch_gemm(0, 0, M, HD, D, 1.f, dy, D, Wout, HD, 0.f, dFbuf, HD, nullptr, gws, GEMM_WS_BYTES, st));
        if (dWout != nullptr)
            GCGCN_TRY(launch_gemm(1, 0, D, HD, M, 1.f, dy, D, F, HD, 0.f, dWout, HD, nullptr, gws, GEMM_WS_BYTES, st));
        if (dbout != nullptr) GCGCN_TRY(launch_colsum(dy, M, D, D, dbout, gws, GEMM_WS_BYTES, st));
        dF = dFbuf;
    }
    if (att_grad == ATT_GRAD_DA)
        GCGCN_TRY(launch_stack_bwd(bt, heads, layers, slab, flags, A, Z, G, Winner, keep, dF, dZ, dE, att_out, frag, st));
    else
        GCGCN_TRY(launch_block_bwd(bt, heads, layers, att_grad, A, q, Z, G, Winner, dF, dZ, dE, att_out, frag, drop, st));
    // dx = [residual: sum_h dF_h] + dZ WnX^T ; debar = dE We^T
    float beta = 0.f;
    if (flags & GCGCN_STACK_RESIDUAL) {
        float* Wsum = (linear && heads > 1 && slab == D && in_dim == D) ? ar.take<float>(static_cast<size_t>(D) * D) : nullptr;
        if (Wsum != nullptr) {
            wout_head_sum_kernel<<<ceil_div(D * D, 256), 256, 0, st>>>(Wout, heads, Wsum);
            GCGCN_CHECK_LAUNCH("wout_head_sum");
            GCGCN_TRY(launch_gemm(0, 0, M, D, D, 1.f, dy, D, Wsum, D, 0.f, dx, D, nullptr, gws, GEMM_WS_BYTES, st));
        } else {
            GCGCN_TRY(launch_head_sum(dF, heads, M, dx, st));
        }
        beta = 1.f;
    }
    GCGCN_TRY(launch_gemm(0, 1, M, in_dim, HD, 1.f, dZ, HD, WnX, HD, beta, dx, in_dim, nullptr, gws, GEMM_WS_BYTES, st));
    GCGCN_TRY(launch_gemm(0, 1, M, D, HD, 1.f, dE, HD, We, HD, 0.f, debar, D, nullptr, gws, GEMM_WS_BYTES, st));
    if (dWnX != nullptr)
        GCGCN_TRY(launch_gemm(1, 0, in_dim, HD, M, 1.f, x, in_dim, dZ, HD, 0.f, dWnX, HD, nullptr, gws, GEMM_WS_BYTES, st));
    if (dWe != nullptr)
        GCGCN_TRY(launch_gemm(1, 0, D, HD, M, 1.f, ebar, D, dE, HD, 0.f, dWe, HD, nullptr, gws, GEMM_WS_BYTES, st));
    if (dWinner != nullptr && layers > 1) {
        GCGCN_TRY(cuda_ok(cudaMemsetAsync(dWinner, 0, static_cast<size_t>(heads) * layers * slab * gd * sizeof(float), st),
                          "memset dWinner"));
        // dWinner[h][l][m*g + k][c] = sum_rows G[row][h*S + m*g + k] * dZ[row][h*S + l*g + c],  m < l
        // (all heads of one sub-layer in a single batched launch)
        for (int l = 1; l < layers; ++l)
            GCGCN_TRY(launch_gemm_batched(1, 0, l * gd, gd, M, 1.f, G, HD, dZ + l * gd, HD, 0.f,
                                          dWinner + static_cast<size_t>(l) * slab * gd, gd, heads, slab, slab,
                                          static_cast<long long>(layers) * slab * gd, gws, GEMM_WS_BYTES, st));
    }
    return GCGCN_OK;
}

int gcgcn_graphconv_stack_bwd(const gcgcn_batch* bt, int32_t heads, int32_t layers, int32_t in_dim,
                              int32_t slab, int32_t flags, const float* x, const float* ebar, const float* A,
                              const float* WnX, const float* We, const float* Winner, const float* Wout,
                              const float* keep, const float* Z, const float* G, const float* F,
                              const float* dy, float* dx, float* debar, float* dA, float* dWnX, float* dWe,
                              float* dWinner, float* dWout, float* dbout, void* ws, size_t ws_bytes,
                              void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_batch(bt));
    GCGCN_REQUIRE(heads >= 1 && layers >= 1 && in_dim >= 1 && slab >= 1 && slab % layers == 0,
                  "stack_bwd: bad heads/layers/widths");
    const bool linear = flags & GCGCN_STACK_LINEAR;
    GCGCN_REQUIRE(linear || heads == 1, "stack_bwd: without the output linear there can be only one head");
    GCGCN_REQUIRE(!(flags & GCGCN_STACK_RESIDUAL) || (in_dim == slab && slab == D),
                  "stack_bwd: the residual needs input width == output width == %d", D);
    if (bt->total_nodes == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(x, "node_feat"));
    GCGCN_TRY(check_device_ptr(A, "adj_matrix"));
    GCGCN_TRY(check_device_ptr(Z, "Z"));
    GCGCN_TRY(check_device_ptr(G, "G"));
    GCGCN_TRY(check_device_ptr(dy, "dy"));
    GCGCN_TRY(check_device_ptr(dx, "dx"));
    GCGCN_TRY(check_device_ptr(debar, "debar"));
    GCGCN_TRY(check_device_ptr(dA, "dA"));
    return stack_bwd_impl(bt, heads, layers, in_dim, slab, flags, ATT_GRAD_DA, x, ebar, A, nullptr, WnX, We, Winner,
                          Wout, keep, Z, G, F, dy, dx, debar, dA, dWnX, dWe, dWinner, dWout, dbout, ws, ws_bytes,
                          static_cast<cudaStream_t>(stream));
}

// ---- dropout stream export (tests) ------------------------------------------------------------
int gcgcn_dropout_mask(uint64_t seed, int32_t stream_id, float p, int64_t count, float* out, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(p >= 0.f && p < 1.f && count >= 0 && stream_id >= 0, "dropout_mask: bad arguments");
    if (count == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(out, "out"));
    return launch_dropout_mask(seed, static_cast<uint32_t>(stream_id), drop_threshold(p), 1.0f / (1.0f - p), count, out,
                               static_cast<cudaStream_t>(stream));
}

// ---- a5 + a6 fused: MultiHeadAttention scores inside the MAGGC block kernels --------------------
int gcgcn_block_supported(const gcgcn_batch* bt, int32_t heads, int32_t layers, int32_t mha) {
    if (bt == nullptr || layers < 1 || D % layers != 0) return 0;
    return block_kernels_usable(bt, heads, layers, D, mha != 0) ? 1 : 0;
}

int gcgcn_mha_stack_fwd(const gcgcn_batch* bt, int32_t heads, int32_t layers, const float* x, const float* ebar,
                        const float* Wq, const float* bq, const float* WnX, const float* We, const float* Winner,
                        const float* Wout, const float* bout, float* q, float* P, float* Z, float* G, float* F,
                        float* y, const gcgcn_dropout* dropout, void* ws, size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_batch(bt));
    BlockDrop drop;
    GCGCN_TRY(make_block_drop(dropout, DROP_STREAM_MHA, DROP_STREAM_MAGGC, &drop));
    GCGCN_REQUIRE(heads >= 1 && layers >= 1 && D % layers == 0, "mha_stack_fwd: bad heads/layers");
    if (!block_kernels_usable(bt, heads, layers, D, true))
        return fail(GCGCN_ERR_UNSUPPORTED, "mha_stack_fwd: needs documents of <= 64 nodes, 2 or 4 sub-layers and 4 or 8 "
                    "heads (got max_nodes %d, layers %d, heads %d); use gcgcn_mha_fwd + gcgcn_graphconv_stack_fwd",
                    bt->max_nodes, layers, heads);
    if (bt->total_nodes == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(x, "node_feat"));
    GCGCN_TRY(check_device_ptr(ebar, "ebar"));
    GCGCN_TRY(check_device_ptr(Wq, "Wq"));
    GCGCN_TRY(check_device_ptr(WnX, "WnX"));
    GCGCN_TRY(check_device_ptr(We, "We"));
    GCGCN_TRY(check_device_ptr(Wout, "Wout"));
    GCGCN_TRY(check_device_ptr(q, "q"));
    GCGCN_TRY(check_device_ptr(P, "P"));
    GCGCN_TRY(check_device_ptr(Z, "Z"));
    GCGCN_TRY(check_device_ptr(G, "G"));
    GCGCN_TRY(check_device_ptr(F, "F"));
    GCGCN_TRY(check_device_ptr(y, "y"));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    GCGCN_TRY(launch_gemm(0, 1, bt->total_nodes, D, D, 1.f, x, D, Wq, D, 0.f, q, D, bq, ws, ws_bytes, st));
    return stack_fwd_impl(bt, heads, layers, D, D, BLOCK_FLAGS_ALL, x, ebar, nullptr, q, P, WnX, We, Winner, Wout, bout,
                          nullptr, Z, G, F, y, ws, ws_bytes, st, drop);
}

int gcgcn_mha_stack_bwd(const gcgcn_batch* bt, int32_t heads, int32_t layers, const float* x, const float* ebar,
                        const float* Wq, const float* WnX, const float* We, const float* Winner, const float* Wout,
                        const float* q, const float* P, const float* Z, const float* G, const float* F,
                        const float* dy, float* dx, float* debar, float* dWq, float* dbq, float* dWnX, float* dWe,
                        float* dWinner, float* dWout, float* dbout, const gcgcn_dropout* dropout, void* ws,
                        size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_batch(bt));
    BlockDrop drop;
    GCGCN_TRY(make_block_drop(dropout, DROP_STREAM_MHA, DROP_STREAM_MAGGC, &drop));
    GCGCN_REQUIRE(heads >= 1 && layers >= 1 && D % layers == 0, "mha_stack_bwd: bad heads/layers");
    if (!block_kernels_usable(bt, heads, layers, D, true))
        return fail(GCGCN_ERR_UNSUPPORTED, "mha_stack_bwd: unsupported configuration (see gcgcn_mha_stack_fwd)");
    if (bt->total_nodes == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(x, "node_feat"));
    GCGCN_TRY(check_device_ptr(q, "q"));
    GCGCN_TRY(check_device_ptr(P, "P"));
    GCGCN_TRY(check_device_ptr(Z, "Z"));
    GCGCN_TRY(check_device_ptr(G, "G"));
    GCGCN_TRY(check_device_ptr(dy, "dy"));
    GCGCN_TRY(check_device_ptr(dx, "dx"));
    GCGCN_TRY(check_device_ptr(debar, "debar"));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    Arena ar(ws, ws_bytes);
    float* dq = ar.take<float>(static_cast<size_t>(bt->total_nodes) * D);
    if (dq == nullptr) return fail(GCGCN_ERR_WORKSPACE, "mha_stack_bwd: workspace too small");
    void* rest = static_cast<char*>(ws) + ar.off;
    const size_t rest_bytes = ws_bytes - ar.off;
    GCGCN_TRY(stack_bwd_impl(bt, heads, layers, D, D, BLOCK_FLAGS_ALL, ATT_GRAD_DQ, x, ebar, P, q, WnX, We, Winner, Wout,
                             nullptr, Z, G, F, dy, dx, debar, dq, dWnX, dWe, dWinner, dWout, dbout, rest, rest_bytes, st,
                             drop));
    // q = x Wq^T + bq :  dx += dq Wq ; dWq = dq^T x ; dbq = colsum(dq)
    Arena ar2(rest, rest_bytes);
    float* gws = ar2.take<float>(GEMM_WS_BYTES / sizeof(float));
    if (gws == nullptr) return fail(GCGCN_ERR_WORKSPACE, "mha_stack_bwd: workspace too small");
    GCGCN_TRY(launch_gemm(0, 0, bt->total_nodes, D, D, 1.f, dq, D, Wq, D, 1.f, dx, D, nullptr, gws, GEMM_WS_BYTES, st));
    if (dWq != nullptr)
        GCGCN_TRY(launch_gemm(1, 0, D, D, bt->total_nodes, 1.f, dq, D, x, D, 0.f, dWq, D, nullptr, gws, GEMM_WS_BYTES, st));
    if (dbq != nullptr) GCGCN_TRY(launch_colsum(dq, bt->total_nodes, D, D, dbq, gws, GEMM_WS_BYTES, st));
    return GCGCN_OK;
}

// ---- parameter packing -----------------------------------------------------------------------
int gcgcn_pack_stack_weights(const void* wn_ptrs, const void* we_ptrs, int32_t heads, int32_t layers, int32_t slab,
                             float* WnX, float* We, float* Winner, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(heads >= 1 && layers >= 1 && slab >= 1 && slab % layers == 0, "pack_stack: bad heads/layers/slab");
    GCGCN_REQUIRE(layers == 1 || Winner != nullptr, "pack_stack: Winner is required when layers > 1");
    GCGCN_TRY(check_device_ptr(wn_ptrs, "wn_ptrs"));
    GCGCN_TRY(check_device_ptr(we_ptrs, "we_ptrs"));
    GCGCN_TRY(check_device_ptr(WnX, "WnX"));
    GCGCN_TRY(check_device_ptr(We, "We"));
    return launch_pack_stack(static_cast<const float* const*>(wn_ptrs), static_cast<const float* const*>(we_ptrs),
                             heads, layers, slab, WnX, We, Winner, static_cast<cudaStream_t>(stream));
}

int gcgcn_unpack_stack_grads(const float* dWnX, const float* dWe, const float* dWinner, int32_t heads,
                             int32_t layers, int32_t slab, float* dwn_flat, float* dwe_flat, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(heads >= 1 && layers >= 1 && slab >= 1 && slab % layers == 0, "unpack_stack: bad heads/layers/slab");
    GCGCN_REQUIRE(layers == 1 || dWinner != nullptr, "unpack_stack: dWinner is required when layers > 1");
    GCGCN_TRY(check_device_ptr(dWnX, "dWnX"));
    GCGCN_TRY(check_device_ptr(dWe, "dWe"));
    GCGCN_TRY(check_device_ptr(dwn_flat, "dwn_flat"));
    GCGCN_TRY(check_device_ptr(dwe_flat, "dwe_flat"));
    return launch_unpack_stack(dWnX, dWe, dWinner, heads, layers, slab, dwn_flat, dwe_flat,
                               static_cast<cudaStream_t>(stream));
}

// ---- parameter collapse / packing of the attention modules ------------------------------------------------
int gcgcn_gat_collapse_fwd(const float* Wh, const float* bh, const float* Wt, const float* bt, const float* Wr,
                           const float* br, const float* w, const float* b, int32_t hid, float* out, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(hid >= 1, "gat_collapse_fwd: hidden_dim < 1");
    const void* ps[] = {Wh, bh, Wt, bt, Wr, br, w, b, out};
    for (const void* p : ps) GCGCN_TRY(check_device_ptr(p, "gat_collapse operand"));
    return launch_gat_collapse_fwd(Wh, bh, Wt, bt, Wr, br, w, b, hid, out, static_cast<cudaStream_t>(stream));
}
int gcgcn_gat_collapse_bwd(const float* Wh, const float* bh, const float* Wt, const float* bt, const float* Wr,
                           const float* br, const float* w, const float* dout, int32_t hid, float* dWh, float* dbh,
                           float* dWt, float* dbt, float* dWr, float* dbr, float* dw, float* db, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(hid >= 1, "gat_collapse_bwd: hidden_dim < 1");
    const void* ps[] = {Wh, bh, Wt, bt, Wr, br, w, dout, dWh, dbh, dWt, dbt, dWr, dbr, dw, db};
    for (const void* p : ps) GCGCN_TRY(check_device_ptr(p, "gat_collapse operand"));
    return launch_gat_collapse_bwd(Wh, bh, Wt, bt, Wr, br, w, dout, hid, dWh, dbh, dWt, dbt, dWr, dbr, dw, db,
                                   static_cast<cudaStream_t>(stream));
}
int gcgcn_pack_rows(const void* ptrs, int32_t count, int32_t elems, float* out, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(count >= 0 && elems >= 0, "pack_rows: negative size");
    if (count == 0 || elems == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(ptrs, "ptrs"));
    GCGCN_TRY(check_device_ptr(out, "out"));
    return launch_pack_rows(static_cast<const float* const*>(ptrs), count, elems, out, static_cast<cudaStream_t>(stream));
}

// ---- a8 pair gathers -------------------------------------------------------------------------
int gcgcn_pair_gather_fwd(const gcgcn_batch* bt, const float* feat, int32_t feat_w, const float* dis,
                          int32_t dis_w, const int32_t* h_idx, const int32_t* t_idx, const int32_t* dis_h,
                          const int32_t* dis_t, float* out_h, float* out_t, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_batch(bt));
    GCGCN_REQUIRE(feat_w > 0 && feat_w % 4 == 0 && dis_w >= 0 && dis_w % 4 == 0,
                  "pair_gather: widths must be multiples of 4 (feat_w=%d, dis_w=%d)", feat_w, dis_w);
    if (bt->total_pairs == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(feat, "feat"));
    GCGCN_TRY(check_device_ptr(h_idx, "h_idx"));
    GCGCN_TRY(check_device_ptr(t_idx, "t_idx"));
    GCGCN_TRY(check_device_ptr(out_h, "out_h"));
    GCGCN_TRY(check_device_ptr(out_t, "out_t"));
    if (dis_w > 0) {
        GCGCN_TRY(check_device_ptr(dis, "dis"));
        GCGCN_TRY(check_device_ptr(dis_h, "dis_h"));
        GCGCN_TRY(check_device_ptr(dis_t, "dis_t"));
    }
    return launch_pair_gather_fwd(bt, feat, feat_w, dis, dis_w, h_idx, t_idx, dis_h, dis_t, out_h, out_t,
                                  static_cast<cudaStream_t>(stream));
}

int gcgcn_pair_gather_bwd(const gcgcn_batch* bt, const float* dout_h, const float* dout_t, int32_t feat_w,
                          int32_t dis_w, int32_t dis_rows, const int32_t* dis_h, const int32_t* dis_t,
                          float* dfeat, float* ddis, void* ws, size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_batch(bt));
    GCGCN_REQUIRE(feat_w > 0 && feat_w % 4 == 0 && dis_w >= 0 && dis_w % 4 == 0,
                  "pair_gather: widths must be multiples of 4 (feat_w=%d, dis_w=%d)", feat_w, dis_w);
    if (bt->total_nodes == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(dout_h, "dout_h"));
    GCGCN_TRY(check_device_ptr(dout_t, "dout_t"));
    GCGCN_TRY(check_device_ptr(dfeat, "dfeat"));
    return launch_pair_gather_bwd(bt, dout_h, dout_t, feat_w, dis_w, dis_rows, dis_h, dis_t, dfeat, ddis, ws,
                                  ws_bytes, static_cast<cudaStream_t>(stream));
}

int gcgcn_pair_dense_fwd(const gcgcn_batch* bt, const float* U, const float* Vd, const int32_t* h_idx,
                         const int32_t* t_idx, const int32_t* dis_h, const int32_t* dis_t, float* out_h, float* out_t,
                         void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_batch(bt));
    if (bt->total_pairs == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(U, "U"));
    GCGCN_TRY(check_device_ptr(Vd, "Vd"));
    GCGCN_TRY(check_device_ptr(h_idx, "h_idx"));
    GCGCN_TRY(check_device_ptr(t_idx, "t_idx"));
    GCGCN_TRY(check_device_ptr(dis_h, "dis_h"));
    GCGCN_TRY(check_device_ptr(dis_t, "dis_t"));
    GCGCN_TRY(check_device_ptr(out_h, "out_h"));
    GCGCN_TRY(check_device_ptr(out_t, "out_t"));
    return launch_pair_dense_fwd(bt, U, Vd, h_idx, t_idx, dis_h, dis_t, out_h, out_t, static_cast<cudaStream_t>(stream));
}

size_t gcgcn_pair_dense_ws_bytes(int32_t dis_rows) {
    return (static_cast<size_t>(pair_dis_warps()) + 4) * dis_rows * D * sizeof(float);
}

int gcgcn_pair_dense_bwd(const gcgcn_batch* bt, const float* dout_h, const float* dout_t, const float* out_h,
                         const float* out_t, int32_t dis_rows, const int32_t* dis_h, const int32_t* dis_t, float* dU,
                         float* dVd, float* dpre, void* ws, size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_batch(bt));
    GCGCN_REQUIRE(dis_rows >= 1, "pair_dense_bwd: dis_rows must be positive");
    if (bt->total_nodes == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(dout_h, "dout_h"));
    GCGCN_TRY(check_device_ptr(dout_t, "dout_t"));
    GCGCN_TRY(check_device_ptr(out_h, "out_h"));
    GCGCN_TRY(check_device_ptr(out_t, "out_t"));
    GCGCN_TRY(check_device_ptr(dU, "dU"));
    GCGCN_TRY(check_device_ptr(dVd, "dVd"));
    GCGCN_TRY(check_device_ptr(dpre, "dpre"));
    return launch_pair_dense_bwd(bt, dout_h, dout_t, out_h, out_t, dis_rows, dis_h, dis_t, dU, dVd, dpre, ws, ws_bytes,
                                 static_cast<cudaStream_t>(stream));
}

// ---- edge-feature producer (SURVEY.md 8f row 1) ------------------------------------------------------------
namespace {
constexpr size_t WT_PARTIAL_FLOATS = 21 * D + D + 4, SP_PARTIAL_FLOATS = D + 4;
int check_edge_tables(const gcgcn_edge_tables* t) {
    if (t == nullptr) return fail(GCGCN_ERR_INVALID_ARG, "edge tables are NULL");
    if (t->num_tokens < 0 || t->num_slots < 0 || t->num_pairs < 0 || t->att_total < 0)
        return fail(GCGCN_ERR_INVALID_ARG, "negative size in edge tables");
    if (t->num_slots > 0) {
        GCGCN_TRY(check_device_ptr(t->slot_tok0, "tabs.slot_tok0"));
        GCGCN_TRY(check_device_ptr(t->slot_len, "tabs.slot_len"));
        GCGCN_TRY(check_device_ptr(t->slot_span, "tabs.slot_span"));
        GCGCN_TRY(check_device_ptr(t->slot_att, "tabs.slot_att"));
    }
    return GCGCN_OK;
}
}  // namespace

size_t gcgcn_edgefeat_ws_bytes(int32_t num_tokens, int32_t att_total, int32_t num_slots, int32_t num_pairs,
                               int64_t total_pairs) {
    size_t a = align256(static_cast<size_t>(word_table_parts(num_tokens)) * WT_PARTIAL_FLOATS * sizeof(float));
    size_t b = align256(static_cast<size_t>(att_total < 0 ? 0 : att_total) * sizeof(float));
    size_t c = align256(static_cast<size_t>(num_slots < 0 ? 0 : num_slots) * 2 * D * sizeof(float)) +
               align256(static_cast<size_t>(sent_pool_parts(num_pairs)) * SP_PARTIAL_FLOATS * sizeof(float));
    size_t d = align256(static_cast<size_t>(edge_colsum_parts(total_pairs < 0 ? 0 : total_pairs)) * D * sizeof(float));
    size_t m = a > b ? a : b;
    if (c > m) m = c;
    if (d > m) m = d;
    return m + (size_t(4) << 20);
}

int gcgcn_word_table_fwd(const float* SF, const float* DF, const float* wa, const float* ba, int32_t tokens, float* T,
                         void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(tokens >= 0, "word_table_fwd: tokens < 0");
    if (tokens == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(SF, "SF"));
    GCGCN_TRY(check_device_ptr(DF, "DF"));
    GCGCN_TRY(check_device_ptr(wa, "wa"));
    GCGCN_TRY(check_device_ptr(ba, "ba"));
    GCGCN_TRY(check_device_ptr(T, "T"));
    return launch_word_table_fwd(SF, DF, wa, ba, tokens, T, static_cast<cudaStream_t>(stream));
}

int gcgcn_word_table_bwd(const float* SF, const float* DF, const float* wa, const float* dT, int32_t tokens, float* dSF,
                         float* dparams, void* ws, size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(tokens >= 0, "word_table_bwd: tokens < 0");
    GCGCN_TRY(check_device_ptr(DF, "DF"));
    GCGCN_TRY(check_device_ptr(wa, "wa"));
    GCGCN_TRY(check_device_ptr(dparams, "dparams"));
    if (tokens > 0) {
        GCGCN_TRY(check_device_ptr(SF, "SF"));
        GCGCN_TRY(check_device_ptr(dT, "dT"));
        GCGCN_TRY(check_device_ptr(dSF, "dSF"));
    }
    Arena ar(ws, ws_bytes);
    float* partial = ar.take<float>(static_cast<size_t>(word_table_parts(tokens)) * WT_PARTIAL_FLOATS);
    if (partial == nullptr) return fail(GCGCN_ERR_WORKSPACE, "word_table_bwd: workspace too small");
    return launch_word_table_bwd(SF, DF, wa, dT, tokens, dSF, dparams, partial, static_cast<cudaStream_t>(stream));
}

int gcgcn_word_pool_fwd(const gcgcn_edge_tables* tabs, const float* T, const float* ctx, float* att, float* cwa,
                        void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_edge_tables(tabs));
    if (tabs->num_slots == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(T, "T"));
    GCGCN_TRY(check_device_ptr(ctx, "ctx"));
    GCGCN_TRY(check_device_ptr(att, "att"));
    GCGCN_TRY(check_device_ptr(cwa, "cwa"));
    return launch_word_pool_fwd(tabs, T, ctx, att, cwa, static_cast<cudaStream_t>(stream));
}

int gcgcn_word_pool_bwd(const gcgcn_edge_tables* tabs, const float* ctx, const float* att, const float* dcwa,
                        float* dctx, float* dT, void* ws, size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_edge_tables(tabs));
    if (tabs->num_slots == 0 || tabs->num_tokens == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(ctx, "ctx"));
    GCGCN_TRY(check_device_ptr(att, "att"));
    GCGCN_TRY(check_device_ptr(dcwa, "dcwa"));
    GCGCN_TRY(check_device_ptr(dctx, "dctx"));
    GCGCN_TRY(check_device_ptr(dT, "dT"));
    GCGCN_TRY(check_device_ptr(tabs->tok_first, "tabs.tok_first"));
    Arena ar(ws, ws_bytes);
    float* dlog = ar.take<float>(static_cast<size_t>(tabs->att_total));
    if (dlog == nullptr) return fail(GCGCN_ERR_WORKSPACE, "word_pool_bwd: workspace too small");
    return launch_word_pool_bwd(tabs, ctx, att, dcwa, dlog, dctx, dT, static_cast<cudaStream_t>(stream));
}

int gcgcn_sent_pool_fwd(const gcgcn_edge_tables* tabs, const float* cw, const float* sfeat, const float* nfeat,
                        const float* va, const float* ca, float* score, float* csa, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_edge_tables(tabs));
    if (tabs->num_pairs == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(cw, "cw"));
    GCGCN_TRY(check_device_ptr(sfeat, "sfeat"));
    GCGCN_TRY(check_device_ptr(nfeat, "nfeat"));
    GCGCN_TRY(check_device_ptr(va, "va"));
    GCGCN_TRY(check_device_ptr(ca, "ca"));
    GCGCN_TRY(check_device_ptr(score, "score"));
    GCGCN_TRY(check_device_ptr(csa, "csa"));
    GCGCN_TRY(check_device_ptr(tabs->pair_slot_ptr, "tabs.pair_slot_ptr"));
    return launch_sent_pool_fwd(tabs, cw, sfeat, nfeat, va, ca, score, csa, static_cast<cudaStream_t>(stream));
}

int gcgcn_sent_pool_bwd(const gcgcn_edge_tables* tabs, int32_t total_nodes, const float* cw, const float* sfeat,
                        const float* nfeat, const float* va, const float* score, const float* dcsa, float* dcw,
                        float* dsfeat, float* dnfeat, float* dparams, void* ws, size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_edge_tables(tabs));
    GCGCN_REQUIRE(total_nodes >= 0, "sent_pool_bwd: total_nodes < 0");
    GCGCN_TRY(check_device_ptr(va, "va"));
    GCGCN_TRY(check_device_ptr(dparams, "dparams"));
    if (total_nodes > 0) {
        GCGCN_TRY(check_device_ptr(dnfeat, "dnfeat"));
        GCGCN_TRY(check_device_ptr(tabs->node_ctr_ptr, "tabs.node_ctr_ptr"));
    }
    if (tabs->num_pairs > 0) {
        GCGCN_TRY(check_device_ptr(cw, "cw"));
        GCGCN_TRY(check_device_ptr(score, "score"));
        GCGCN_TRY(check_device_ptr(dcsa, "dcsa"));
        GCGCN_TRY(check_device_ptr(dcw, "dcw"));
        GCGCN_TRY(check_device_ptr(dsfeat, "dsfeat"));
    }
    Arena ar(ws, ws_bytes);
    float* dpre = ar.take<float>(static_cast<size_t>(tabs->num_slots) * 2 * D + 4);
    float* partial = ar.take<float>(static_cast<size_t>(sent_pool_parts(tabs->num_pairs)) * SP_PARTIAL_FLOATS);
    if (dpre == nullptr || partial == nullptr) return fail(GCGCN_ERR_WORKSPACE, "sent_pool_bwd: workspace too small");
    return launch_sent_pool_bwd(tabs, total_nodes, cw, sfeat, nfeat, va, score, dcsa, dcw, dsfeat, dnfeat, dparams, dpre,
                                partial, static_cast<cudaStream_t>(stream));
}

int gcgcn_edge_fill_fwd(const float* bias, const float* rows, const int64_t* pair_idx, int32_t num_pairs,
                        int64_t total_pairs, int32_t edge_dtype, void* e, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(num_pairs >= 0 && total_pairs >= 0, "edge_fill_fwd: negative size");
    if (total_pairs == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(bias, "bias"));
    GCGCN_TRY(check_device_ptr(e, "e"));
    if (num_pairs > 0) {
        GCGCN_TRY(check_device_ptr(rows, "rows"));
        GCGCN_TRY(check_device_ptr(pair_idx, "pair_idx"));
    }
    return launch_edge_fill_fwd(bias, rows, pair_idx, num_pairs, total_pairs, edge_dtype, e, static_cast<cudaStream_t>(stream));
}

int gcgcn_edge_fill_bwd(const void* de, const int64_t* pair_idx, int32_t num_pairs, int64_t total_pairs,
                        int32_t edge_dtype, float* drows, float* dbias, void* ws, size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(num_pairs >= 0 && total_pairs >= 0, "edge_fill_bwd: negative size");
    GCGCN_TRY(check_device_ptr(dbias, "dbias"));
    if (total_pairs > 0) GCGCN_TRY(check_device_ptr(de, "de"));
    if (num_pairs > 0) {
        GCGCN_TRY(check_device_ptr(drows, "drows"));
        GCGCN_TRY(check_device_ptr(pair_idx, "pair_idx"));
    }
    Arena ar(ws, ws_bytes);
    float* partial = ar.take<float>(static_cast<size_t>(edge_colsum_parts(total_pairs)) * D);
    if (partial == nullptr) return fail(GCGCN_ERR_WORKSPACE, "edge_fill_bwd: workspace too small");
    return launch_edge_fill_bwd(de, pair_idx, num_pairs, total_pairs, edge_dtype, drows, dbias, partial,
                                static_cast<cudaStream_t>(stream));
}

int gcgcn_colsum(const float* X, int32_t M, int32_t N, int32_t ldx, float* out, void* ws, size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(M >= 0 && N >= 0 && ldx >= N, "colsum: bad shape");
    if (N == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(out, "out"));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (M == 0) return cuda_ok(cudaMemsetAsync(out, 0, static_cast<size_t>(N) * sizeof(float), st), "colsum: memset");
    GCGCN_TRY(check_device_ptr(X, "X"));
    return launch_colsum(X, M, N, ldx, out, ws, ws_bytes, st);
}

// ---- relation classifier and loss (SURVEY.md 8f row 2) -----------------------------------------------------
int gcgcn_bilinear_reduce_fwd(const float* Y, const float* t, const float* bias, int32_t rows, int32_t relations,
                              int32_t accumulate, float* out, int32_t ldo, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(rows >= 0 && relations >= 0 && ldo >= relations, "bilinear_reduce: bad shape");
    if (rows == 0 || relations == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(Y, "Y"));
    GCGCN_TRY(check_device_ptr(t, "t"));
    GCGCN_TRY(check_device_ptr(out, "out"));
    return launch_bilinear_reduce(Y, t, bias, rows, relations, accumulate, out, ldo, static_cast<cudaStream_t>(stream));
}
size_t gcgcn_bilinear_ws_bytes(int32_t rows, int32_t relations) {
    const size_t r = static_cast<size_t>(relations < 0 ? 0 : relations), m = static_cast<size_t>(rows < 0 ? 0 : rows);
    const size_t ld = (m + 31) & ~size_t(31);
    return align256(r * 4 * 33024) + align256(2 * r * ld * sizeof(float)) + 4096;      // pre-split W' blobs + partials
}

int gcgcn_bilinear_fwd(const float* h, const float* t, const float* Wm, const float* bias, int32_t rows,
                       int32_t relations, int32_t accumulate, float* out, int32_t ldo, void* ws, size_t ws_bytes,
                       void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(rows >= 0 && relations >= 0 && ldo >= relations, "bilinear_fwd: bad shape");
    if (rows == 0 || relations == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(h, "h"));
    GCGCN_TRY(check_device_ptr(t, "t"));
    GCGCN_TRY(check_device_ptr(Wm, "Wm"));
    GCGCN_TRY(check_device_ptr(out, "out"));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    Arena ar(ws, ws_bytes);
    const size_t ld = (static_cast<size_t>(rows) + 31) & ~size_t(31);
    uint8_t* blobs = ar.take<uint8_t>(static_cast<size_t>(relations) * 4 * 33024);
    float* part = ar.take<float>(2 * static_cast<size_t>(relations) * ld);
    if (blobs == nullptr || part == nullptr) return fail(GCGCN_ERR_WORKSPACE, "bilinear_fwd: workspace too small");
    GCGCN_TRY(launch_gemm_rowop(1, rows, relations * D, D, h, D, Wm, relations * D, t, part, static_cast<long long>(ld), blobs,
                                static_cast<size_t>(relations) * 4 * 33024, st));
    return launch_bilinear_finish(part, static_cast<long long>(ld), bias, rows, relations, accumulate, out, ldo, st);
}

size_t gcgcn_bilinear_bwd_ws_bytes(int32_t rows, int32_t relations) {
    const size_t r = static_cast<size_t>(relations < 0 ? 0 : relations);
    // pre-split W' blobs, one [128, relations*128] partial per 4096-row range of the weight-gradient GEMM, pre-split h
    const size_t ranges = (static_cast<size_t>(rows < 0 ? 0 : rows) + 4095) / 4096;
    return align256(r * 4 * 33024) + align256(std::max<size_t>(GEMM_WS_BYTES, ranges * D * r * D * sizeof(float))) +
           align256(gemm_presplit_bytes(rows < 0 ? 0 : rows)) + 4096;
}

int gcgcn_bilinear_bwd(const float* h, const float* t, const float* Wm, const float* Wm2, const float* dout, int32_t rows,
                       int32_t relations, float beta, float* dh, float* dt, float* dWm, void* ws, size_t ws_bytes,
                       void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(rows >= 0 && relations >= 1, "bilinear_bwd: bad shape");
    if (rows < 8192)
        return fail(GCGCN_ERR_UNSUPPORTED, "bilinear_bwd: the fused backward needs >= 8192 rows (got %d); use "
                    "gcgcn_bilinear_outer_bwd / gcgcn_bilinear_dt_bwd with gcgcn_gemm", rows);
    const void* ps[] = {h, t, Wm, Wm2, dout, dh, dt, dWm};
    for (const void* p : ps) GCGCN_TRY(check_device_ptr(p, "bilinear_bwd operand"));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    Arena ar(ws, ws_bytes);
    const size_t blob_bytes = static_cast<size_t>(relations) * 4 * 33024, pre_bytes = gemm_presplit_bytes(rows);
    const size_t ranges = (static_cast<size_t>(rows) + 4095) / 4096;
    const size_t gws_bytes = std::max<size_t>(GEMM_WS_BYTES, ranges * D * static_cast<size_t>(relations) * D * sizeof(float));
    uint8_t* blobs = ar.take<uint8_t>(blob_bytes);
    uint8_t* gws = ar.take<uint8_t>(gws_bytes);
    uint8_t* pre = ar.take<uint8_t>(pre_bytes);
    if (blobs == nullptr || gws == nullptr || pre == nullptr)
        return fail(GCGCN_ERR_WORKSPACE, "bilinear_bwd: workspace too small");
    const int N = relations * D;
    GCGCN_TRY(launch_gemm_rowop(2, rows, N, D, h, D, Wm, N, dout, dt, relations, blobs, blob_bytes, st));
    GCGCN_TRY(launch_gemm_rowop(2, rows, N, D, t, D, Wm2, N, dout, dh, relations, blobs, blob_bytes, st));
    return launch_gemm_wgrad_scaled(D, relations, rows, h, D, t, dout, relations, beta, dWm, N, gws, gws_bytes, st, pre,
                                    pre_bytes);
}

int gcgcn_bilinear_outer_bwd(const float* dout, int32_t ldd, const float* t, int32_t rows, int32_t relations, float* dY,
                             void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(rows >= 0 && relations >= 0 && ldd >= relations, "bilinear_outer: bad shape");
    if (rows == 0 || relations == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(dout, "dout"));
    GCGCN_TRY(check_device_ptr(t, "t"));
    GCGCN_TRY(check_device_ptr(dY, "dY"));
    return launch_bilinear_outer(dout, ldd, t, rows, relations, dY, static_cast<cudaStream_t>(stream));
}
int gcgcn_bilinear_dt_bwd(const float* dout, int32_t ldd, const float* Y, int32_t rows, int32_t relations, float* dt,
                          void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(rows >= 0 && relations >= 0 && ldd >= relations, "bilinear_dt: bad shape");
    if (rows == 0 || relations == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(dout, "dout"));
    GCGCN_TRY(check_device_ptr(Y, "Y"));
    GCGCN_TRY(check_device_ptr(dt, "dt"));
    return launch_bilinear_dt(dout, ldd, Y, rows, relations, dt, static_cast<cudaStream_t>(stream));
}
int gcgcn_doc_bias_fwd(const gcgcn_batch* bt, const float* v, int32_t relations, float* z, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_batch(bt));
    GCGCN_REQUIRE(relations >= 1, "doc_bias_fwd: relations < 1");
    if (bt->total_pairs == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(v, "v"));
    GCGCN_TRY(check_device_ptr(z, "z"));
    return launch_doc_bias_fwd(bt, v, relations, z, static_cast<cudaStream_t>(stream));
}
int gcgcn_doc_bias_bwd(const gcgcn_batch* bt, const float* dz, int32_t relations, float* dv, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_batch(bt));
    GCGCN_REQUIRE(relations >= 1, "doc_bias_bwd: relations < 1");
    if (bt->num_docs == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(dv, "dv"));
    if (bt->total_pairs > 0) GCGCN_TRY(check_device_ptr(dz, "dz"));
    return launch_doc_bias_bwd(bt, dz, relations, dv, static_cast<cudaStream_t>(stream));
}
int gcgcn_pair_bce_fwd(const gcgcn_batch* bt, const float* logits, const float* labels, int32_t relations, float* loss,
                       void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_batch(bt));
    GCGCN_REQUIRE(relations >= 1, "pair_bce_fwd: relations < 1");
    if (bt->num_docs == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(loss, "loss"));
    if (bt->total_pairs > 0) {
        GCGCN_TRY(check_device_ptr(logits, "logits"));
        GCGCN_TRY(check_device_ptr(labels, "labels"));
    }
    return launch_pair_bce_fwd(bt, logits, labels, relations, loss, static_cast<cudaStream_t>(stream));
}
int gcgcn_pair_bce_bwd(const gcgcn_batch* bt, const float* logits, const float* labels, int32_t relations,
                       const float* dloss, float* dlogits, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_batch(bt));
    GCGCN_REQUIRE(relations >= 1, "pair_bce_bwd: relations < 1");
    if (bt->total_pairs == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(logits, "logits"));
    GCGCN_TRY(check_device_ptr(labels, "labels"));
    GCGCN_TRY(check_device_ptr(dloss, "dloss"));
    GCGCN_TRY(check_device_ptr(dlogits, "dlogits"));
    return launch_pair_bce_bwd(bt, logits, labels, relations, dloss, dlogits, static_cast<cudaStream_t>(stream));
}

// ---- relation evaluation ---------------------------------------------------------------------
size_t gcgcn_rank_ws_bytes(int64_t count) { return rank_ws_bytes(count); }
int gcgcn_rank_candidates(const gcgcn_batch* bt, const float* logits, int32_t relations, const float* labels,
                          const uint8_t* intrain, int64_t base_id, float* score, uint32_t* payload, int64_t* counters,
                          void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_batch(bt));
    GCGCN_REQUIRE(relations >= 2, "rank_candidates: relations < 2 (relation 0 is not a candidate)");
    GCGCN_REQUIRE(base_id >= 0, "rank_candidates: negative base_id");
    const long long count = (bt->total_pairs - bt->total_nodes) * static_cast<long long>(relations - 1);
    GCGCN_REQUIRE(count >= 0, "rank_candidates: total_pairs < total_nodes");
    if (base_id + count >= GCGCN_RANK_MAX_CANDIDATES)
        return fail(GCGCN_ERR_UNSUPPORTED, "rank_candidates: %lld + %lld candidates, one evaluation holds fewer than 2^30",
                    static_cast<long long>(base_id), count);
    GCGCN_TRY(check_device_ptr(counters, "counters"));
    if (count == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(logits, "logits"));
    if (labels != nullptr) GCGCN_TRY(check_device_ptr(labels, "labels"));
    if (intrain != nullptr) GCGCN_TRY(check_device_ptr(intrain, "intrain"));
    GCGCN_TRY(check_device_ptr(score, "score"));
    GCGCN_TRY(check_device_ptr(payload, "payload"));
    return launch_rank_candidates(bt, logits, labels, intrain, relations, base_id, score, payload,
                                  reinterpret_cast<unsigned long long*>(counters), static_cast<cudaStream_t>(stream));
}
int gcgcn_rank_candidates_at(const gcgcn_batch* bt, const float* logits, int32_t relations, const float* labels,
                             const uint8_t* intrain, const int64_t* doc_base, float* score, uint32_t* payload,
                             int64_t* counters, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_batch(bt));
    GCGCN_REQUIRE(relations >= 2, "rank_candidates_at: relations < 2 (relation 0 is not a candidate)");
    const long long count = (bt->total_pairs - bt->total_nodes) * static_cast<long long>(relations - 1);
    GCGCN_REQUIRE(count >= 0, "rank_candidates_at: total_pairs < total_nodes");
    if (count >= GCGCN_RANK_MAX_CANDIDATES)
        return fail(GCGCN_ERR_UNSUPPORTED, "rank_candidates_at: %lld candidates, one evaluation holds fewer than 2^30",
                    count);
    GCGCN_TRY(check_device_ptr(counters, "counters"));
    if (count == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(logits, "logits"));
    if (labels != nullptr) GCGCN_TRY(check_device_ptr(labels, "labels"));
    if (intrain != nullptr) GCGCN_TRY(check_device_ptr(intrain, "intrain"));
    GCGCN_TRY(check_device_ptr(doc_base, "doc_base"));
    GCGCN_TRY(check_device_ptr(score, "score"));
    GCGCN_TRY(check_device_ptr(payload, "payload"));
    return launch_rank_candidates_at(bt, logits, labels, intrain, relations, reinterpret_cast<const long long*>(doc_base),
                                     score, payload, reinterpret_cast<unsigned long long*>(counters),
                                     static_cast<cudaStream_t>(stream));
}
int gcgcn_rank_sort(const float* score, const uint32_t* payload, int64_t count, uint32_t* sorted_key,
                    uint32_t* sorted_payload, void* ws, size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(count >= 0 && count < GCGCN_RANK_MAX_CANDIDATES, "rank_sort: count %lld outside [0, 2^30)",
                  static_cast<long long>(count));
    if (count == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(score, "score"));
    GCGCN_TRY(check_device_ptr(payload, "payload"));
    GCGCN_TRY(check_device_ptr(sorted_key, "sorted_key"));
    GCGCN_TRY(check_device_ptr(sorted_payload, "sorted_payload"));
    GCGCN_TRY(check_device_ptr(ws, "ws"));
    GCGCN_REQUIRE(ws_bytes >= rank_ws_bytes(count), "rank_sort: ws_bytes %zu < gcgcn_rank_ws_bytes = %zu", ws_bytes,
                  rank_ws_bytes(count));
    return launch_rank_sort(score, payload, count, sorted_key, sorted_payload, ws, ws_bytes,
                            static_cast<cudaStream_t>(stream));
}
int gcgcn_rank_curve(const uint32_t* sorted_key, const uint32_t* sorted_payload, int64_t count, int64_t total_recall,
                     int32_t has_intrain, double input_theta, gcgcn_rank_result* result, void* ws, size_t ws_bytes,
                     void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(count >= 1 && count < GCGCN_RANK_MAX_CANDIDATES, "rank_curve: count %lld outside [1, 2^30)",
                  static_cast<long long>(count));
    GCGCN_TRY(check_device_ptr(sorted_key, "sorted_key"));
    GCGCN_TRY(check_device_ptr(sorted_payload, "sorted_payload"));
    GCGCN_REQUIRE((reinterpret_cast<uintptr_t>(sorted_payload) & 15) == 0, "rank_curve: sorted_payload not 16-byte aligned");
    GCGCN_TRY(check_device_ptr(result, "result"));
    GCGCN_TRY(check_device_ptr(ws, "ws"));
    GCGCN_REQUIRE(ws_bytes >= rank_ws_bytes(count), "rank_curve: ws_bytes %zu < gcgcn_rank_ws_bytes = %zu", ws_bytes,
                  rank_ws_bytes(count));
    return launch_rank_curve(sorted_key, sorted_payload, count, total_recall < 1 ? 1 : total_recall, has_intrain ? 1 : 0,
                             input_theta, result, ws, ws_bytes, static_cast<cudaStream_t>(stream));
}
size_t gcgcn_rank_merge_ws_bytes(int64_t count) { return rank_merge_ws_bytes(count); }
int gcgcn_rank_merge(const uint32_t* key_a, const uint32_t* payload_a, int64_t na, const uint32_t* key_b,
                     const uint32_t* payload_b, int64_t nb, uint32_t* key_out, uint32_t* payload_out, void* ws,
                     size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(na >= 0 && nb >= 0, "rank_merge: negative run length");
    GCGCN_REQUIRE(na + nb < GCGCN_RANK_MAX_CANDIDATES, "rank_merge: %lld + %lld candidates, one evaluation holds fewer than 2^30",
                  static_cast<long long>(na), static_cast<long long>(nb));
    if (na + nb == 0) return GCGCN_OK;
    if (na > 0) {
        GCGCN_TRY(check_device_ptr(key_a, "key_a"));
        GCGCN_TRY(check_device_ptr(payload_a, "payload_a"));
    }
    if (nb > 0) {
        GCGCN_TRY(check_device_ptr(key_b, "key_b"));
        GCGCN_TRY(check_device_ptr(payload_b, "payload_b"));
    }
    GCGCN_TRY(check_device_ptr(key_out, "key_out"));
    GCGCN_TRY(check_device_ptr(payload_out, "payload_out"));
    GCGCN_REQUIRE(((reinterpret_cast<uintptr_t>(key_out) | reinterpret_cast<uintptr_t>(payload_out)) & 15) == 0,
                  "rank_merge: key_out / payload_out not 16-byte aligned");
    GCGCN_TRY(check_device_ptr(ws, "ws"));
    GCGCN_REQUIRE(ws_bytes >= rank_merge_ws_bytes(na + nb), "rank_merge: ws_bytes %zu < gcgcn_rank_merge_ws_bytes = %zu",
                  ws_bytes, rank_merge_ws_bytes(na + nb));
    return launch_rank_merge(key_a, payload_a, na, key_b, payload_b, nb, key_out, payload_out, ws, ws_bytes,
                             static_cast<cudaStream_t>(stream));
}
int gcgcn_rank_curve_points(const uint32_t* sorted_payload, int64_t count, int64_t total_recall, int32_t has_intrain,
                            float* x, float* y, float* y_ign, void* ws, size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(count >= 1 && count < GCGCN_RANK_MAX_CANDIDATES, "rank_curve_points: count %lld outside [1, 2^30)",
                  static_cast<long long>(count));
    GCGCN_TRY(check_device_ptr(sorted_payload, "sorted_payload"));
    GCGCN_REQUIRE((reinterpret_cast<uintptr_t>(sorted_payload) & 15) == 0,
                  "rank_curve_points: sorted_payload not 16-byte aligned");
    GCGCN_TRY(check_device_ptr(x, "x"));
    GCGCN_TRY(check_device_ptr(y, "y"));
    if (has_intrain) GCGCN_TRY(check_device_ptr(y_ign, "y_ign"));
    GCGCN_TRY(check_device_ptr(ws, "ws"));
    GCGCN_REQUIRE(ws_bytes >= rank_ws_bytes(count), "rank_curve_points: ws_bytes %zu < gcgcn_rank_ws_bytes = %zu",
                  ws_bytes, rank_ws_bytes(count));
    return launch_rank_curve_points(sorted_payload, count, total_recall < 1 ? 1 : total_recall, has_intrain ? 1 : 0, x,
                                    y, y_ign, ws, ws_bytes, static_cast<cudaStream_t>(stream));
}
int gcgcn_rank_decode(const uint32_t* sorted_key, const uint32_t* sorted_payload, int64_t rows, int64_t count,
                      const int64_t* doc_offsets, const int32_t* doc_n, int32_t num_docs, int32_t relations, int32_t* doc,
                      int32_t* row, int32_t* col, int32_t* relation, float* score, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(rows >= 0 && num_docs >= 1 && relations >= 2, "rank_decode: bad shape");
    GCGCN_REQUIRE(rows <= count, "rank_decode: rows %lld > count %lld of the ranking", static_cast<long long>(rows),
                  static_cast<long long>(count));
    if (rows == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(sorted_key, "sorted_key"));
    GCGCN_TRY(check_device_ptr(sorted_payload, "sorted_payload"));
    GCGCN_TRY(check_device_ptr(doc_offsets, "doc_offsets"));
    GCGCN_TRY(check_device_ptr(doc_n, "doc_n"));
    GCGCN_TRY(check_device_ptr(doc, "doc"));
    GCGCN_TRY(check_device_ptr(row, "row"));
    GCGCN_TRY(check_device_ptr(col, "col"));
    GCGCN_TRY(check_device_ptr(relation, "relation"));
    GCGCN_TRY(check_device_ptr(score, "score"));
    return launch_rank_decode(sorted_key, sorted_payload, rows, reinterpret_cast<const long long*>(doc_offsets), doc_n,
                              num_docs, relations, doc, row, col, relation, score, static_cast<cudaStream_t>(stream));
}

// ---- relation evaluation per relation --------------------------------------------------------------------------
// count in [1, 2^30), a multiple of R - 1, and R - 1 <= 256 (one 8-bit digit)
static int check_relations(const char* what, int64_t count, int32_t relations) {
    if (relations < 2) return fail(GCGCN_ERR_INVALID_ARG, "%s: relations < 2 (relation 0 is not a candidate)", what);
    if (relations - 1 > 256)
        return fail(GCGCN_ERR_UNSUPPORTED, "%s: %d relations r >= 1, at most 256 (one 8-bit digit)", what,
                    relations - 1);
    if (count < 1 || count >= GCGCN_RANK_MAX_CANDIDATES)
        return fail(GCGCN_ERR_INVALID_ARG, "%s: count %lld outside [1, 2^30)", what, static_cast<long long>(count));
    if (count % (relations - 1) != 0)
        return fail(GCGCN_ERR_INVALID_ARG, "%s: count %lld is not a multiple of relations - 1 = %d", what,
                    static_cast<long long>(count), relations - 1);
    return GCGCN_OK;
}
static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

size_t gcgcn_rank_relations_ws_bytes(int64_t count, int32_t relations) {
    return rank_relations_ws_bytes(count, relations);
}
int gcgcn_rank_by_relation(const uint32_t* sorted_key, const uint32_t* sorted_payload, int64_t count, int32_t relations,
                           uint32_t* rel_key, uint32_t* rel_payload, void* ws, size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_relations("rank_by_relation", count, relations));
    GCGCN_TRY(check_device_ptr(sorted_key, "sorted_key"));
    GCGCN_TRY(check_device_ptr(sorted_payload, "sorted_payload"));
    GCGCN_TRY(check_device_ptr(rel_key, "rel_key"));
    GCGCN_TRY(check_device_ptr(rel_payload, "rel_payload"));
    GCGCN_TRY(check_device_ptr(ws, "ws"));
    GCGCN_REQUIRE(ws_bytes >= rank_relations_ws_bytes(count, relations),
                  "rank_by_relation: ws_bytes %zu < gcgcn_rank_relations_ws_bytes = %zu", ws_bytes,
                  rank_relations_ws_bytes(count, relations));
    return launch_rank_by_relation(sorted_key, sorted_payload, count, relations, rel_key, rel_payload, ws, ws_bytes,
                                   static_cast<cudaStream_t>(stream));
}
int gcgcn_rank_curve_relations(const uint32_t* rel_key, const uint32_t* rel_payload, int64_t count, int32_t relations,
                               const int64_t* total_recall, int32_t has_intrain, const double* input_theta,
                               gcgcn_rank_result* results, void* ws, size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_relations("rank_curve_relations", count, relations));
    GCGCN_TRY(check_device_ptr(rel_key, "rel_key"));
    GCGCN_TRY(check_device_ptr(rel_payload, "rel_payload"));
    GCGCN_REQUIRE(aligned16(rel_payload), "rank_curve_relations: rel_payload not 16-byte aligned");
    if (total_recall != nullptr) GCGCN_TRY(check_device_ptr(total_recall, "total_recall"));
    GCGCN_TRY(check_device_ptr(input_theta, "input_theta"));
    GCGCN_TRY(check_device_ptr(results, "results"));
    GCGCN_TRY(check_device_ptr(ws, "ws"));
    GCGCN_REQUIRE(ws_bytes >= rank_relations_ws_bytes(count, relations),
                  "rank_curve_relations: ws_bytes %zu < gcgcn_rank_relations_ws_bytes = %zu", ws_bytes,
                  rank_relations_ws_bytes(count, relations));
    return launch_rank_curve_relations(rel_key, rel_payload, count, relations,
                                       reinterpret_cast<const long long*>(total_recall), has_intrain ? 1 : 0,
                                       input_theta, results, ws, ws_bytes, static_cast<cudaStream_t>(stream));
}
int gcgcn_rank_select(const uint32_t* sorted_key, const uint32_t* sorted_payload, int64_t count, int32_t relations,
                      const float* theta, uint32_t* out_key, uint32_t* out_payload, int64_t* counts, void* ws,
                      size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_TRY(check_relations("rank_select", count, relations));
    GCGCN_TRY(check_device_ptr(sorted_key, "sorted_key"));
    GCGCN_TRY(check_device_ptr(sorted_payload, "sorted_payload"));
    GCGCN_REQUIRE(aligned16(sorted_key) && aligned16(sorted_payload), "rank_select: inputs not 16-byte aligned");
    GCGCN_TRY(check_device_ptr(theta, "theta"));
    GCGCN_TRY(check_device_ptr(out_key, "out_key"));
    GCGCN_TRY(check_device_ptr(out_payload, "out_payload"));
    GCGCN_TRY(check_device_ptr(counts, "counts"));
    GCGCN_TRY(check_device_ptr(ws, "ws"));
    GCGCN_REQUIRE(ws_bytes >= rank_relations_ws_bytes(count, relations),
                  "rank_select: ws_bytes %zu < gcgcn_rank_relations_ws_bytes = %zu", ws_bytes,
                  rank_relations_ws_bytes(count, relations));
    return launch_rank_select(sorted_key, sorted_payload, count, relations, theta, out_key, out_payload,
                              reinterpret_cast<long long*>(counts), ws, ws_bytes, static_cast<cudaStream_t>(stream));
}

// ---- dense projection ------------------------------------------------------------------------
int gcgcn_expand_pair_context(const int32_t* slots, int32_t num_slots, int32_t n, int32_t max_num, int32_t length,
                              int32_t dis_plus, uint8_t* sen_matrix, int64_t* pos_matrix_h, int64_t* pos_matrix_t,
                              void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(num_slots >= 0 && n >= 0 && max_num >= 0 && length >= 0, "expand_pair_context: negative size");
    if (static_cast<size_t>(n) * n * max_num * length == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(sen_matrix, "sen_matrix"));
    GCGCN_TRY(check_device_ptr(pos_matrix_h, "pos_matrix_h"));
    GCGCN_TRY(check_device_ptr(pos_matrix_t, "pos_matrix_t"));
    if (num_slots > 0) GCGCN_TRY(check_device_ptr(slots, "slots"));
    return launch_expand_pair_context(slots, num_slots, n, max_num, length, dis_plus, sen_matrix,
                                      reinterpret_cast<long long*>(pos_matrix_h),
                                      reinterpret_cast<long long*>(pos_matrix_t), static_cast<cudaStream_t>(stream));
}

int gcgcn_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t count,
                    float lr, float beta1, float beta2, float eps, float weight_decay, float grad_scale,
                    int32_t step, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(count >= 0 && step >= 1, "adam_step: count >= 0 and step >= 1 required");
    GCGCN_REQUIRE(beta1 >= 0.f && beta1 < 1.f && beta2 >= 0.f && beta2 < 1.f && eps > 0.f, "adam_step: bad betas/eps");
    if (count == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(params, "params"));
    GCGCN_TRY(check_device_ptr(grads, "grads"));
    GCGCN_TRY(check_device_ptr(exp_avg, "exp_avg"));
    GCGCN_TRY(check_device_ptr(exp_avg_sq, "exp_avg_sq"));
    GCGCN_REQUIRE(((reinterpret_cast<uintptr_t>(params) | reinterpret_cast<uintptr_t>(grads) |
                    reinterpret_cast<uintptr_t>(exp_avg) | reinterpret_cast<uintptr_t>(exp_avg_sq)) & 15) == 0,
                  "adam_step: buffers must be 16-byte aligned");
    return launch_adam(params, grads, exp_avg, exp_avg_sq, count, lr, beta1, beta2, eps, weight_decay, grad_scale,
                       step, static_cast<cudaStream_t>(stream));
}

int gcgcn_gemm(int32_t ta, int32_t tb, int32_t M, int32_t N, int32_t K, float alpha, const float* A,
               int32_t lda, const float* B, int32_t ldb, float beta, float* C, int32_t ldc, const float* bias,
               void* ws, size_t ws_bytes, void* stream) {
    GCGCN_API_ENTER(stream);
    GCGCN_REQUIRE(M >= 0 && N >= 0 && K >= 0, "gemm: negative dimension");
    if (M == 0 || N == 0) return GCGCN_OK;
    GCGCN_TRY(check_device_ptr(C, "C"));
    if (K > 0) {
        GCGCN_TRY(check_device_ptr(A, "A"));
        GCGCN_TRY(check_device_ptr(B, "B"));
    }
    // only the first GEMM_WS_BYTES of ws are used (split-K partials / pre-split weight blobs).  The split-K count and the
    // choice of kernel depend on the size passed; the cap keeps them independent of how large a workspace the caller has
    const size_t head = ws_bytes < GEMM_WS_BYTES ? ws_bytes : GEMM_WS_BYTES;
    return launch_gemm(ta, tb, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, bias, ws, head,
                       static_cast<cudaStream_t>(stream));
}

// ---- block-level composites ------------------------------------------------------------------
namespace {
struct CagSaved { float *P, *ebar, *Z, *G, *F; };
struct MagSaved { float *ebar, *q, *P, *Z, *G, *F; };

CagSaved carve_cag(void* saved, int nodes, long long pairs) {
    Arena ar(saved, ~size_t(0) >> 1);
    CagSaved s;
    s.P = ar.take<float>(pairs);
    s.ebar = ar.take<float>(static_cast<size_t>(nodes) * D);
    s.Z = ar.take<float>(static_cast<size_t>(nodes) * D);
    s.G = ar.take<float>(static_cast<size_t>(nodes) * D);
    s.F = ar.take<float>(static_cast<size_t>(nodes) * D);
    return s;
}
MagSaved carve_mag(void* saved, int nodes, long long pairs, int heads) {
    Arena ar(saved, ~size_t(0) >> 1);
    MagSaved s;
    s.ebar = ar.take<float>(static_cast<size_t>(nodes) * D);
    s.q = ar.take<float>(static_cast<size_t>(nodes) * D);
    s.P = ar.take<float>(static_cast<size_t>(pairs) * heads);
    s.Z = ar.take<float>(static_cast<size_t>(nodes) * heads * D);
    s.G = ar.take<float>(static_cast<size_t>(nodes) * heads * D);
    s.F = ar.take<float>(static_cast<size_t>(nodes) * heads * D);
    return s;
}
constexpr int BLOCK_FLAGS = GCGCN_STACK_RELU | GCGCN_STACK_RESIDUAL | GCGCN_STACK_LINEAR;
}  // namespace

size_t gcgcn_block_saved_bytes(int32_t total_nodes, int64_t total_pairs, int32_t heads) {
    const size_t nodes = static_cast<size_t>(total_nodes), h = static_cast<size_t>(heads < 1 ? 1 : heads);
    return align256(static_cast<size_t>(total_pairs) * h * sizeof(float)) +
           2 * align256(nodes * D * sizeof(float)) + 3 * align256(nodes * h * D * sizeof(float)) + 1024;
}

int gcgcn_caggc_fwd(const gcgcn_batch* bt, int32_t layers, const float* x, const void* e, int32_t edge_dtype,
                    const float* u, const float* v, const float* c, const float* WnX, const float* We,
                    const float* Winner, const float* Wout, const float* bout, float* y, void* saved,
                    const gcgcn_dropout* dropout, void* ws, size_t ws_bytes, void* stream) {
    ::gcgcn::StreamDeviceGuard outer_guard__(static_cast<cudaStream_t>(stream));   // composite: covers its own launches too
    GCGCN_TRY(check_batch(bt));
    GCGCN_TRY(check_device_ptr(saved, "saved"));
    BlockDrop drop;
    GCGCN_TRY(make_block_drop(dropout, DROP_STREAM_GAT, DROP_STREAM_CAGGC, &drop));
    CagSaved s = carve_cag(saved, bt->total_nodes, bt->total_pairs);
    // s.P = the GAT softmax output; with dropout the block kernel applies the (regenerated) keep mask to it
    GCGCN_TRY(gcgcn_gat_fwd(bt, x, e, edge_dtype, u, v, c, nullptr, 0, nullptr, s.P, s.P, s.ebar, ws, ws_bytes, stream));
    if (!drop_active(drop))
        return gcgcn_graphconv_stack_fwd(bt, 1, layers, D, D, BLOCK_FLAGS, x, s.ebar, s.P, WnX, We, Winner, Wout, bout,
                                         nullptr, s.Z, s.G, s.F, y, ws, ws_bytes, stream);
    if (!block_kernels_usable(bt, 1, layers, D, false))
        return fail(GCGCN_ERR_UNSUPPORTED, "caggc_fwd: in-kernel dropout needs documents of <= 64 nodes and 2 or 4 "
                    "sub-layers; pass keep masks through gcgcn_gat_fwd / gcgcn_graphconv_stack_fwd instead");
    GCGCN_API_ENTER(stream);
    return stack_fwd_impl(bt, 1, layers, D, D, BLOCK_FLAGS, x, s.ebar, s.P, nullptr, nullptr, WnX, We, Winner, Wout, bout,
                          nullptr, s.Z, s.G, s.F, y, ws, ws_bytes, static_cast<cudaStream_t>(stream), drop);
}

int gcgcn_caggc_bwd(const gcgcn_batch* bt, int32_t layers, const float* x, const void* e, int32_t edge_dtype,
                    const float* u, const float* v, const float* WnX, const float* We, const float* Winner,
                    const float* Wout, const float* dy, const void* saved, float* dx, void* de, float* du,
                    float* dv, float* dc, float* dWnX, float* dWe, float* dWinner, float* dWout, float* dbout,
                    const gcgcn_dropout* dropout, void* ws, size_t ws_bytes, void* stream) {
    ::gcgcn::StreamDeviceGuard outer_guard__(static_cast<cudaStream_t>(stream));   // composite: covers its own launches too
    GCGCN_TRY(check_batch(bt));
    GCGCN_TRY(check_device_ptr(saved, "saved"));
    BlockDrop drop;
    GCGCN_TRY(make_block_drop(dropout, DROP_STREAM_GAT, DROP_STREAM_CAGGC, &drop));
    CagSaved s = carve_cag(const_cast<void*>(saved), bt->total_nodes, bt->total_pairs);
    // tail of the workspace holds the gradients that flow between the two halves of the block
    Arena ar(ws, ws_bytes);
    float* dx_stack = ar.take<float>(static_cast<size_t>(bt->total_nodes) * D);
    float* debar = ar.take<float>(static_cast<size_t>(bt->total_nodes) * D);
    float* dA = ar.take<float>(bt->total_pairs);
    if (dx_stack == nullptr || debar == nullptr || dA == nullptr)
        return fail(GCGCN_ERR_WORKSPACE, "caggc_bwd: workspace too small");
    void* rest = static_cast<char*>(ws) + ar.off;
    const size_t rest_bytes = ws_bytes - ar.off;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (block_kernels_usable(bt, 1, layers, D, false)) {
        // the block kernel finishes the softmax backward in shared memory: dA never exists in HBM
        float* dS = dA;
        GCGCN_API_ENTER(stream);
        GCGCN_TRY(stack_bwd_impl(bt, 1, layers, D, D, BLOCK_FLAGS, ATT_GRAD_DS, x, s.ebar, s.P, nullptr, WnX, We, Winner,
                                 Wout, nullptr, s.Z, s.G, s.F, dy, dx_stack, debar, dS, dWnX, dWe, dWinner, dWout, dbout,
                                 rest, rest_bytes, st, drop));
        Arena ar2(rest, rest_bytes);
        GCGCN_TRY(gat_bwd_from_ds(bt, x, e, edge_dtype, u, v, dS, debar, dx, de, du, dv, dc, ar2, st));
    } else {
        if (drop_active(drop)) return fail(GCGCN_ERR_UNSUPPORTED, "caggc_bwd: in-kernel dropout needs the block kernels");
        GCGCN_TRY(gcgcn_graphconv_stack_bwd(bt, 1, layers, D, D, BLOCK_FLAGS, x, s.ebar, s.P, WnX, We, Winner, Wout,
                                            nullptr, s.Z, s.G, s.F, dy, dx_stack, debar, dA, dWnX, dWe, dWinner, dWout,
                                            dbout, rest, rest_bytes, stream));
        GCGCN_TRY(gcgcn_gat_bwd(bt, x, e, edge_dtype, u, v, nullptr, 0, nullptr, s.P, dA, debar, dx, de, du, dv, dc,
                                rest, rest_bytes, stream));
    }
    return launch_add(dx, dx_stack, static_cast<size_t>(bt->total_nodes) * D, st);
}

int gcgcn_maggc_fwd(const gcgcn_batch* bt, int32_t layers, int32_t heads, const float* x, const void* e,
                    int32_t edge_dtype, const float* Wq, const float* bq, const float* WnX, const float* We,
                    const float* Winner, const float* Wout, const float* bout, float* y, void* saved,
                    const gcgcn_dropout* dropout, void* ws, size_t ws_bytes, void* stream) {
    ::gcgcn::StreamDeviceGuard outer_guard__(static_cast<cudaStream_t>(stream));   // composite: covers its own launches too
    GCGCN_TRY(check_batch(bt));
    GCGCN_TRY(check_device_ptr(saved, "saved"));
    MagSaved s = carve_mag(saved, bt->total_nodes, bt->total_pairs, heads);
    GCGCN_TRY(gcgcn_edge_mean_fwd(bt, e, edge_dtype, s.ebar, stream));
    if (block_kernels_usable(bt, heads, layers, D, true))
        return gcgcn_mha_stack_fwd(bt, heads, layers, x, s.ebar, Wq, bq, WnX, We, Winner, Wout, bout, s.q, s.P, s.Z, s.G,
                                   s.F, y, dropout, ws, ws_bytes, stream);
    GCGCN_REQUIRE(dropout == nullptr || (dropout->p_att <= 0.f && dropout->p_gcn <= 0.f),
                  "maggc_fwd: in-kernel dropout needs the block kernels (n <= 64, 4 or 8 heads)");
    GCGCN_TRY(gcgcn_mha_fwd(bt, heads, x, Wq, bq, nullptr, s.q, s.P, s.P, ws, ws_bytes, stream));
    return gcgcn_graphconv_stack_fwd(bt, heads, layers, D, D, BLOCK_FLAGS, x, s.ebar, s.P, WnX, We, Winner, Wout, bout,
                                     nullptr, s.Z, s.G, s.F, y, ws, ws_bytes, stream);
}

int gcgcn_maggc_bwd(const gcgcn_batch* bt, int32_t layers, int32_t heads, const float* x, int32_t edge_dtype,
                    const float* Wq, const float* WnX, const float* We, const float* Winner, const float* Wout,
                    const float* dy, const void* saved, float* dx, void* de, float* dWq, float* dbq, float* dWnX,
                    float* dWe, float* dWinner, float* dWout, float* dbout, const gcgcn_dropout* dropout, void* ws,
                    size_t ws_bytes, void* stream) {
    ::gcgcn::StreamDeviceGuard outer_guard__(static_cast<cudaStream_t>(stream));   // composite: covers its own launches too
    GCGCN_TRY(check_batch(bt));
    GCGCN_TRY(check_device_ptr(saved, "saved"));
    MagSaved s = carve_mag(const_cast<void*>(saved), bt->total_nodes, bt->total_pairs, heads);
    Arena ar(ws, ws_bytes);
    float* dx_stack = ar.take<float>(static_cast<size_t>(bt->total_nodes) * D);
    float* debar = ar.take<float>(static_cast<size_t>(bt->total_nodes) * D);
    float* dA = ar.take<float>(static_cast<size_t>(bt->total_pairs) * heads);
    if (dx_stack == nullptr || debar == nullptr || dA == nullptr)
        return fail(GCGCN_ERR_WORKSPACE, "maggc_bwd: workspace too small");
    void* rest = static_cast<char*>(ws) + ar.off;
    const size_t rest_bytes = ws_bytes - ar.off;
    if (block_kernels_usable(bt, heads, layers, D, true)) {
        GCGCN_TRY(gcgcn_mha_stack_bwd(bt, heads, layers, x, s.ebar, Wq, WnX, We, Winner, Wout, s.q, s.P, s.Z, s.G, s.F, dy,
                                      dx, debar, dWq, dbq, dWnX, dWe, dWinner, dWout, dbout, dropout, rest, rest_bytes,
                                      stream));
        return gcgcn_edge_mean_bwd(bt, debar, edge_dtype, de, stream);
    }
    GCGCN_REQUIRE(dropout == nullptr || (dropout->p_att <= 0.f && dropout->p_gcn <= 0.f),
                  "maggc_bwd: in-kernel dropout needs the block kernels (n <= 64, 4 or 8 heads)");
    GCGCN_TRY(gcgcn_graphconv_stack_bwd(bt, heads, layers, D, D, BLOCK_FLAGS, x, s.ebar, s.P, WnX, We, Winner, Wout,
                                        nullptr, s.Z, s.G, s.F, dy, dx_stack, debar, dA, dWnX, dWe, dWinner,
                                        dWout, dbout, rest, rest_bytes, stream));
    GCGCN_TRY(gcgcn_mha_bwd(bt, heads, x, Wq, s.q, nullptr, s.P, dA, dx, dWq, dbq, rest, rest_bytes, stream));
    GCGCN_TRY(launch_add(dx, dx_stack, static_cast<size_t>(bt->total_nodes) * D, static_cast<cudaStream_t>(stream)));
    return gcgcn_edge_mean_bwd(bt, debar, edge_dtype, de, stream);
}

}  // extern "C"
