/*
 * gcgcn_b200 -- C ABI of the B200-native (sm_100a) entity-graph convolution hot path of GCGCN.
 *
 * The reference (Huiweizhou/GCGCN) has no FFI: its boundary for this path is the Python
 * nn.Module surface in models/GCGCN_glove.py (G) and
 * models/GraphCNN_multihead_bert_gate_cls.py (B; graph classes byte-identical to G).  Every
 * entry point below therefore cites the reference *method* it replaces.  The Python drop-in
 * modules in gcgcn_b200/modules.py bind these symbols with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the comment says "host"; a CPU buffer is an
 *     error, never a fallback;
 *   - the library never allocates or frees: outputs, saved-for-backward buffers and
 *     workspaces are caller-owned (sizes via the *_workspace_bytes functions);
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); nothing synchronises;
 *   - return value: 0 = ok, negative = error (see codes); gcgcn_last_error() gives the text
 *     for the calling thread;
 *   - node-sized tensors ([total_nodes, *]) and attention maps are float32; the n x n x 128
 *     edge tensors (the bytes that matter) are float32 or bfloat16, selected by `edge_dtype`;
 *     accumulation is always float32;
 *   - hidden width d = 128 (G:234) is a compile-time constant of the kernels.
 *
 * Ragged batches: B document graphs are concatenated.  Node rows of document b live at
 * [node_ptr[b], node_ptr[b+1]); its n_b x n_b pair grid (edge features, attention maps,
 * masks) starts at pair offset pair_ptr[b] (= sum of n^2 of earlier documents) and is
 * row-major [i][j].  B = 1 reproduces the reference's un-batched call.
 */
#ifndef GCGCN_B200_H
#define GCGCN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GCGCN_HIDDEN 128

#define GCGCN_OK 0
#define GCGCN_ERR_INVALID_ARG (-1)
#define GCGCN_ERR_UNSUPPORTED (-2)
#define GCGCN_ERR_CUDA (-3)
#define GCGCN_ERR_WORKSPACE (-4)

#define GCGCN_F32 0
#define GCGCN_BF16 1

/* flags of gcgcn_graphconv_stack_{fwd,bwd} */
#define GCGCN_STACK_RELU 1       /* relu after every sub-layer (G:71, G:108)                    */
#define GCGCN_STACK_RESIDUAL 2   /* F_h = cat_l drop(g_l) + x  (G:75-76, G:112-113)             */
#define GCGCN_STACK_LINEAR 4     /* y = Linear(cat_h F_h)      (G:78, G:117-118)                */

#define GCGCN_TILE_ROWS 96

typedef struct gcgcn_batch {
    int32_t num_docs;        /* B                                                        */
    int32_t total_nodes;     /* sum_b n_b                                                */
    int64_t total_pairs;     /* sum_b n_b^2                                              */
    int32_t max_nodes;       /* max_b n_b                                                */
    int32_t reserved;
    const int32_t* node_ptr; /* [B+1] device                                             */
    const int64_t* pair_ptr; /* [B+1] device                                             */
    const int32_t* row_doc;  /* [total_nodes] device: document of each node row          */
    /* optional scheduling hint (may be NULL / zeros): documents sorted by n descending, and how
     * many of them have n > 48, n > 32, n > 16 and n > 0.  Lets the per-document kernels launch one
     * grid per size class with right-sized shared memory instead of sizing every CTA for max_nodes. */
    const int32_t* doc_order; /* [B] device                                              */
    int32_t class_end[4];     /* cumulative counts in doc_order: n>48, n>32, n>16, n>0   */
    /* optional packing hint (may be NULL / 0): consecutive documents grouped into tiles of at most tile_rows
     * (= GCGCN_TILE_ROWS) node rows, tile t = documents [tile_doc[t], tile_doc[t+1]).  Lets the MAGGC block run on
     * packed tensor-core tiles (csrc/gcn_tile.cu) instead of one CTA per document; absent (or a document with more
     * entities than a tile holds) -> the per-document kernels. */
    const int32_t* tile_doc;  /* [num_tiles+1] device                                    */
    int32_t num_tiles;
    int32_t tile_rows;
} gcgcn_batch;

/* ---- train-mode dropout of the block-level entry points ------------------------------------------
 * The reference drops attention probabilities (nn.Dropout(0.1), G:131, G:152 -> G:141, G:166) and each
 * sub-layer's output copy (gcn_dropout 0.2, G:59, G:90 -> G:74, G:108).  The block kernels regenerate the
 * keep-scale factors (0 or 1/(1-p)) from (seed, stream, element index) with a counter-based hash in forward AND
 * backward, so no mask tensor exists; gcgcn_dropout_mask materialises a stream (tests compare this route with
 * the keep-mask-in route of gcgcn_gat_fwd / gcgcn_mha_fwd / gcgcn_graphconv_stack_fwd element for element).
 * Streams: 1 GAT attention [pairs], 2 CAGGC sub-layer outputs [rows*128], 3 MHA attention [heads*pairs],
 * 4 MAGGC sub-layer outputs [rows*heads*128]; element index = row-major offset in that tensor.
 * A NULL pointer (or both probabilities 0) means no dropout.                                       */
typedef struct gcgcn_dropout {
    uint64_t seed;
    float p_att;    /* attention dropout probability, in [0, 1) */
    float p_gcn;    /* sub-layer output dropout probability, in [0, 1) */
} gcgcn_dropout;
int gcgcn_dropout_mask(uint64_t seed, int32_t stream_id, float p, int64_t count, float* out, void* stream);

/* ---- library ---------------------------------------------------------------------------- */
const char* gcgcn_version(void);
const char* gcgcn_last_error(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
uint64_t gcgcn_launch_count(void);
/* Packed-tile tensor-core path of the MAGGC block (csrc/gcn_tile.cu): 1 = use it where its preconditions hold,
 * 0 = per-document kernels everywhere.  Returns the previous setting; initially on unless the environment variable
 * GCGCN_TILE_BLOCKS is 0.  Both paths compute the same function (fp32 rounding apart). */
int32_t gcgcn_set_tile_blocks(int32_t enable);
/* fills SM count and compute capability of the current device */
int gcgcn_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor);
/* per-kernel timing for bench.py: begin() starts recording one CUDA event after every launch on
 * `stream`; end() synchronises and writes "<kernel>\t<launches>\t<total ms>\t<total flop>\n" lines
 * into buf (flop: 2MNK summed over the launches of the dense-projection kernels, 0 for the others). */
int gcgcn_timing_begin(void* stream);
int gcgcn_timing_end(void* stream, char* buf, size_t cap);
/* upper bound, in bytes, of the workspace any entry point below needs for this batch shape */
size_t gcgcn_workspace_bytes(int32_t total_nodes, int64_t total_pairs, int32_t heads);

/* ---- a1: mention->entity pooling, replaces G:297-298 (= B:287-288) ------------------------
 * x0[e,:] = sum_k w[k] * ctx[tok_idx[k],:] for k in [ent_ptr[e], ent_ptr[e+1]).
 * The CSR table is built on the host bit-exactly from the reference's node_pos weights
 * (config/Config.py:169-176, 223) by gcgcn_b200.batch.PoolTable.
 * bwd uses the transposed table (token -> entities) so it is a deterministic gather too.   */
int gcgcn_pool_fwd(const float* ctx, const int32_t* ent_ptr, const int32_t* tok_idx, const float* w,
                   int32_t total_nodes, float* x0, void* stream);
int gcgcn_pool_bwd(const float* dx0, const int32_t* tok_ptr, const int32_t* ent_idx, const float* w_t,
                   int32_t total_tokens, float* dctx, void* stream);

/* ---- shared edge pass ("K_edge_reduce"), the n^2*d stream of G:40-41 and G:161 ----------
 * mean only (what GraphConv needs from the edge tensor, G:40-41 collapsed):
 *   ebar[r,:] = mean_j e[i,j,:]                      r = node row of (b,i)
 * bwd: de[i,j,:] = debar[r,:] / n_b                                                        */
int gcgcn_edge_mean_fwd(const gcgcn_batch* bt, const void* e, int32_t edge_dtype, float* ebar,
                        void* stream);
int gcgcn_edge_mean_bwd(const gcgcn_batch* bt, const float* debar, int32_t edge_dtype, void* de,
                        void* stream);

/* ---- a2: GATAttention.forward(node_feat, edge_feat, mask), replaces G:154-168 -------------
 * energy_ij = u.x_j + v.e_ij + c  with  u = Wh^T w1 + Wt^T w2, v = Wr^T w3,
 * c = w1.bh + w2.bt + w3.br + b (exact collapse of G:156-162; built from the reference-named
 * parameters on the host side); P = softmax_j(energy); A = P * keep.
 * mask: uint8 [total_pairs], honoured only if apply_mask != 0 (the reference ignores it,
 * G:163-164).  keep: keep-scale dropout mask [total_pairs] (0 or 1/(1-p)) or NULL (eval).
 * The same pass over e also yields ebar for the following GraphConvolution.
 * fwd outputs: P (softmax), A (post-dropout; may alias P when keep == NULL), ebar.
 * ws: >= total_nodes floats.                                                               */
int gcgcn_gat_fwd(const gcgcn_batch* bt, const float* x, const void* e, int32_t edge_dtype,
                  const float* u, const float* v, const float* c, const uint8_t* mask,
                  int32_t apply_mask, const float* keep, float* P, float* A, float* ebar,
                  void* ws, size_t ws_bytes, void* stream);
/* bwd inputs: dA (grad of A), debar (grad of ebar, may be NULL).
 * outputs: dx [total_nodes,128], de (edge_dtype) [total_pairs,128], du[128], dv[128], dc[1]. */
int gcgcn_gat_bwd(const gcgcn_batch* bt, const float* x, const void* e, int32_t edge_dtype,
                  const float* u, const float* v, const uint8_t* mask, int32_t apply_mask,
                  const float* keep, const float* P, const float* dA, const float* debar,
                  float* dx, void* de, float* du, float* dv, float* dc,
                  void* ws, size_t ws_bytes, void* stream);

/* ---- a5: MultiHeadAttention.forward(node_feat, mask=None), replaces G:133-142 -------------
 * q = x Wq^T + bq (Wq = the H linears_q weights stacked to [128,128], G:129);
 * P_h = softmax(q_h q_h^T / sqrt(d_h)) -- the key uses linears_q too (G:137);
 * A_h = P_h * keep_h.  Attention maps are head-major: [H][total_pairs].
 * q [total_nodes,128] is an output saved for backward.                                     */
int gcgcn_mha_fwd(const gcgcn_batch* bt, int32_t heads, const float* x, const float* Wq,
                  const float* bq, const float* keep, float* q, float* P, float* A,
                  void* ws, size_t ws_bytes, void* stream);
int gcgcn_mha_bwd(const gcgcn_batch* bt, int32_t heads, const float* x, const float* Wq,
                  const float* q, const float* keep, const float* P, const float* dA,
                  float* dx, float* dWq, float* dbq, void* ws, size_t ws_bytes, void* stream);

/* ---- a3/a4/a6: GraphConv / GraphConvolution / MultiGraphConvolution .forward -------------
 * replaces G:36-50, G:63-80, G:97-120.  For head h and sub-layer l (g = 128 / layers):
 *   Z_hl = x WnX[:, h,l] + sum_{m<l} g_hm Winner[h,l,m]        (node projection, dense connect)
 *   out  = ( ebar We[:, h,l] + A_h Z_hl ) / r_h ,  r = rowsum(A_h) + [rowsum == 0]  (G:43-50)
 *   g_hl = relu(out);  F_h = cat_l(keep * g_hl) + x;  y = cat_h(F_h) Wout^T + bout
 * Packed weights (built by the drop-in modules from the reference-named parameters):
 *   WnX  [128, H*128]  column h*128 + l*g + c  = graphconv[h*L+l].weights_node[0:128, c]
 *   We   [128, H*128]  column h*128 + l*g + c  = graphconv[h*L+l].weights_edge[:, c]
 *   Winner [H][L][128][g]  row m*g + k (m < l) = graphconv[h*L+l].weights_node[128 + m*g + k, :]
 *   Wout [128, H*128], bout [128]              = linear_layer.{weight,bias}
 * A: [H][total_pairs]; keep: [total_nodes, H*128] or NULL.
 * Saved for backward (caller-owned, float32): Z, G, F -- each [total_nodes, H*128].
 * flags: GCGCN_STACK_*; without GCGCN_STACK_LINEAR, y receives F (H must be 1 then).
 * in_dim = width of x (rows of WnX), slab = per-head output width = layers * g.  Inside the two
 * conv blocks both are 128; a stand-alone GraphConv(input_dim, 128, output_dim) (G:19) is
 * layers = 1, in_dim = input_dim, slab = output_dim in {16,32,64,128}, flags = 0, and every
 * "H*128" above reads "H*slab".                                                            */
int gcgcn_graphconv_stack_fwd(const gcgcn_batch* bt, int32_t heads, int32_t layers, int32_t in_dim,
                              int32_t slab, int32_t flags,
                              const float* x, const float* ebar, const float* A,
                              const float* WnX, const float* We, const float* Winner,
                              const float* Wout, const float* bout, const float* keep,
                              float* Z, float* G, float* F, float* y,
                              void* ws, size_t ws_bytes, void* stream);
int gcgcn_graphconv_stack_bwd(const gcgcn_batch* bt, int32_t heads, int32_t layers, int32_t in_dim,
                              int32_t slab, int32_t flags,
                              const float* x, const float* ebar, const float* A,
                              const float* WnX, const float* We, const float* Winner,
                              const float* Wout, const float* keep,
                              const float* Z, const float* G, const float* F, const float* dy,
                              float* dx, float* debar, float* dA,
                              float* dWnX, float* dWe, float* dWinner, float* dWout, float* dbout,
                              void* ws, size_t ws_bytes, void* stream);

/* ---- a5 + a6 fused: MultiHeadAttention inside the MAGGC block kernels (G:133-142 + G:97-120) ----
 * Inference / no-dropout form of  adj = MultiHeadAttention(x) ; y = MultiGraphConvolution(x, e, adj)
 * (the reference's call pair at G:336-337) for documents of <= 64 entities, layer_num 2 or 4 and
 * head_num 4 or 8 -- gcgcn_block_supported(bt, heads, layers, 1) says whether a batch qualifies
 * (mha = 0 asks the same for a given attention map, i.e. the CAGGC block).  The softmax of
 * q_h q_h^T / sqrt(d_h) is taken inside the per-(document, head) kernel that consumes it and, in the
 * backward, the softmax gradient and dq are finished there too: no [H][sum n^2] array is re-read.
 * q [total_nodes,128] and P [heads][total_pairs] are outputs of fwd (saved for bwd; P is the
 * attention list the reference would return); Z, G, F, dx, debar and the parameter gradients are as
 * in gcgcn_graphconv_stack_*.  ebar = gcgcn_edge_mean_fwd(e); the caller sends debar through
 * gcgcn_edge_mean_bwd.                                                                        */
int gcgcn_block_supported(const gcgcn_batch* bt, int32_t heads, int32_t layers, int32_t mha);
int gcgcn_mha_stack_fwd(const gcgcn_batch* bt, int32_t heads, int32_t layers,
                        const float* x, const float* ebar, const float* Wq, const float* bq,
                        const float* WnX, const float* We, const float* Winner,
                        const float* Wout, const float* bout,
                        float* q, float* P, float* Z, float* G, float* F, float* y,
                        const gcgcn_dropout* dropout, void* ws, size_t ws_bytes, void* stream);
int gcgcn_mha_stack_bwd(const gcgcn_batch* bt, int32_t heads, int32_t layers,
                        const float* x, const float* ebar, const float* Wq,
                        const float* WnX, const float* We, const float* Winner, const float* Wout,
                        const float* q, const float* P, const float* Z, const float* G,
                        const float* F, const float* dy,
                        float* dx, float* debar, float* dWq, float* dbq,
                        float* dWnX, float* dWe, float* dWinner, float* dWout, float* dbout,
                        const gcgcn_dropout* dropout, void* ws, size_t ws_bytes, void* stream);

/* ---- parameter packing for the stack entry points ----------------------------------------
 * The reference keeps one weights_node [128 + l*g, g] and one weights_edge [128, g] per GraphConv
 * (G:24-25, heads*layers of them).  pack gathers them (device arrays of heads*layers device pointers,
 * GraphConv index k = h*layers + l) into WnX / We / Winner in one launch; unpack scatters the packed
 * gradients into two flat buffers holding the per-GraphConv gradients back to back in index order.   */
int gcgcn_pack_stack_weights(const void* wn_ptrs, const void* we_ptrs, int32_t heads, int32_t layers,
                             int32_t slab, float* WnX, float* We, float* Winner, void* stream);
int gcgcn_unpack_stack_grads(const float* dWnX, const float* dWe, const float* dWinner, int32_t heads,
                             int32_t layers, int32_t slab, float* dwn_flat, float* dwe_flat, void* stream);

/* ---- a2 parameter collapse: the eight GATAttention parameters -> (u, v, c) of gcgcn_gat_fwd, and back ------------
 * Wh/Wt/Wr = linear_node_h / linear_node_t / linear_edge_r .weight [hid, 128], bh/bt/br their biases [hid],
 * w = wt.weight [3*hid], b = wt.bias [1].  out = [u (128) | v (128) | c (1)];  bwd takes dout in the same layout.   */
int gcgcn_gat_collapse_fwd(const float* Wh, const float* bh, const float* Wt, const float* bt, const float* Wr,
                           const float* br, const float* w, const float* b, int32_t hid, float* out, void* stream);
int gcgcn_gat_collapse_bwd(const float* Wh, const float* bh, const float* Wt, const float* bt, const float* Wr,
                           const float* br, const float* w, const float* dout, int32_t hid, float* dWh, float* dbh,
                           float* dWt, float* dbt, float* dWr, float* dbr, float* dw, float* db, void* stream);
/* out[i] = *ptrs[i] for `count` equally sized float arrays of `elems` elements (ptrs: device array of device pointers):
 * MultiHeadAttention's per-head query projections -> Wq [128,128] / bq [128] (G:129)                                */
int gcgcn_pack_rows(const void* ptrs, int32_t count, int32_t elems, float* out, void* stream);

/* ---- a8: pair gathers, replaces G:351-352 (+ G:306-307) -----------------------------------
 * out_h[p,:] = cat(feat[h_idx[p],:], dis[dis_h[p],:]),  out_t[p,:] = cat(feat[t_idx[p],:], dis[dis_t[p],:])
 * for every pair p of the batch.  Index tables are int32 [total_pairs] holding *global* node
 * rows (h_idx[i,j] = node_ptr[b]+j, t_idx[i,j] = node_ptr[b]+i, quirk 6) and distance rows
 * (dis_plus +/- node_relative_pos), built by gcgcn_b200.batch.PairTables.
 * h_idx / t_idx MUST be these canonical tables: the backward derives the same layout from the batch descriptor
 * instead of reading them (segmented sums over the rows / columns of each pair grid), so any other table would get a
 * forward/backward mismatch.  Every dis_h / dis_t entry must lie in [0, dis_rows): the host builder checks it
 * (PairTables.check_dis_rows); the kernels do not.
 * feat_w and dis_w must be multiples of 4; dis_w may be 0 (in-loop gathers, G:321-322).
 * bwd: dfeat[r,:] = sum over pairs that gathered row r (segmented, deterministic);
 *      ddis[k,:]  = sum over pairs that gathered distance row k.                           */
int gcgcn_pair_gather_fwd(const gcgcn_batch* bt, const float* feat, int32_t feat_w,
                          const float* dis, int32_t dis_w, const int32_t* h_idx,
                          const int32_t* t_idx, const int32_t* dis_h, const int32_t* dis_t,
                          float* out_h, float* out_t, void* stream);
int gcgcn_pair_gather_bwd(const gcgcn_batch* bt, const float* dout_h, const float* dout_t,
                          int32_t feat_w, int32_t dis_w, int32_t dis_rows,
                          const int32_t* dis_h, const int32_t* dis_t,
                          float* dfeat, float* ddis, void* ws, size_t ws_bytes, void* stream);

/* ---- classifier-side pair features without the gathered intermediate (SURVEY.md 8f row 2, first half) ----
 * Replaces G:351-355: entity_feature_h[i,j] = tanh(dense_layer(cat(F[j], dis[10 + rp_ij]))) = tanh(U[j] + Vd[10 + rp_ij])
 * and entity_feature_t[i,j] = tanh(U[i] + Vd[10 - rp_ij]), with U = F W_F^T [total_nodes, 128] and
 * Vd = dis_embed W_d^T + bias [dis_rows, 128] (dense_layer.weight split by input columns; both computed by the caller,
 * node-level work).  Index tables as for gcgcn_pair_gather_fwd.  out_h / out_t: [total_pairs, 128].
 * bwd: dU, dVd = segmented sums of dout (1 - out^2) (deterministic); dpre is caller-owned scratch of
 * 2 * total_pairs * 128 floats, ws of gcgcn_pair_dense_ws_bytes(dis_rows) bytes.                                  */
int gcgcn_pair_dense_fwd(const gcgcn_batch* bt, const float* U, const float* Vd, const int32_t* h_idx,
                         const int32_t* t_idx, const int32_t* dis_h, const int32_t* dis_t, float* out_h, float* out_t,
                         void* stream);
size_t gcgcn_pair_dense_ws_bytes(int32_t dis_rows);
int gcgcn_pair_dense_bwd(const gcgcn_batch* bt, const float* dout_h, const float* dout_t, const float* out_h,
                         const float* out_t, int32_t dis_rows, const int32_t* dis_h, const int32_t* dis_t, float* dU,
                         float* dVd, float* dpre, void* ws, size_t ws_bytes, void* stream);

/* ---- block-level composites (SURVEY.md section 8b minimum set) ---------------------------
 * CAGGC = a2 + a4 sharing one pass over e0 (G:330-333); MAGGC = a5 + a6 (G:336-337).
 * They call the entry points above in order with buffers carved from `ws`; `saved` is a
 * caller-owned arena of gcgcn_block_saved_bytes(...) bytes that bwd reads back.  `dropout`
 * (NULL = none) must be the same struct in fwd and bwd; it needs the block kernels
 * (gcgcn_block_supported), otherwise GCGCN_ERR_UNSUPPORTED is returned.                    */
size_t gcgcn_block_saved_bytes(int32_t total_nodes, int64_t total_pairs, int32_t heads);
int gcgcn_caggc_fwd(const gcgcn_batch* bt, int32_t layers, const float* x, const void* e,
                    int32_t edge_dtype, const float* u, const float* v, const float* c,
                    const float* WnX, const float* We, const float* Winner, const float* Wout,
                    const float* bout, float* y, void* saved, const gcgcn_dropout* dropout,
                    void* ws, size_t ws_bytes, void* stream);
int gcgcn_caggc_bwd(const gcgcn_batch* bt, int32_t layers, const float* x, const void* e,
                    int32_t edge_dtype, const float* u, const float* v,
                    const float* WnX, const float* We, const float* Winner, const float* Wout,
                    const float* dy, const void* saved, float* dx, void* de,
                    float* du, float* dv, float* dc, float* dWnX, float* dWe, float* dWinner,
                    float* dWout, float* dbout, const gcgcn_dropout* dropout,
                    void* ws, size_t ws_bytes, void* stream);
int gcgcn_maggc_fwd(const gcgcn_batch* bt, int32_t layers, int32_t heads, const float* x,
                    const void* e, int32_t edge_dtype, const float* Wq, const float* bq,
                    const float* WnX, const float* We, const float* Winner, const float* Wout,
                    const float* bout, float* y, void* saved, const gcgcn_dropout* dropout,
                    void* ws, size_t ws_bytes, void* stream);
int gcgcn_maggc_bwd(const gcgcn_batch* bt, int32_t layers, int32_t heads, const float* x,
                    int32_t edge_dtype, const float* Wq,
                    const float* WnX, const float* We, const float* Winner, const float* Wout,
                    const float* dy, const void* saved, float* dx, void* de,
                    float* dWq, float* dbq, float* dWnX, float* dWe, float* dWinner,
                    float* dWout, float* dbout, const gcgcn_dropout* dropout,
                    void* ws, size_t ws_bytes, void* stream);

/* ---- wire format -> dense pair-context tensors (SURVEY.md 8f row 3; replaces the host loops of
 * config/Config.py:180-205 and the H2D copies of C:345-347) --------------------------------------------
 * `slots` is int32 [num_slots, 9], one row per (edge, sentence slot) of ONE document:
 * (u, v, slot, s0, s1, h0, h1, t0, t1) = entity pair, slot index, sentence tokens [s0, s1), head and tail
 * mention spans.  Writes sen_matrix (bool as uint8), pos_matrix_h and pos_matrix_t (int64), each
 * [n, n, max_num, length] row-major, exactly as C:219-222 leaves them (rows with slot >= max_num and tokens
 * >= length are truncated away; everything outside the listed spans is 0).  The call zero-fills the outputs. */
int gcgcn_expand_pair_context(const int32_t* slots, int32_t num_slots, int32_t n, int32_t max_num, int32_t length,
                              int32_t dis_plus, uint8_t* sen_matrix, int64_t* pos_matrix_h, int64_t* pos_matrix_t,
                              void* stream);

/* ---- edge-feature producer (SURVEY.md 8f row 1): WordAttention + SentenceAttention as G:299-327 uses them ----
 * Replaces, per hop i, word_attention[i] (G:313-314), linear_word_att[i] (G:317), sentence_attention[i] (G:323-324) and
 * linear_sentence_att[i] (G:326) for a ragged batch of documents.  Only "active" slots are evaluated: a sentence slot
 * whose sentence contains token 0 (sent_att_padding_matrix = ~sen_matrix[:, :, :, 0:1], G:302); every other slot is
 * masked to -1e5 before the relu of G:212, contributes exactly 0 to context_sent_att and receives exactly zero
 * gradient, and a pair without active slots gets linear_sentence_att.bias.  The word scores come from the table
 * T[l][k] = attention_all(tanh(attention_sent(ctx[l]) + attention_pos(dis_embed[k]))) (G:179-183 has 21 L distinct
 * values, not n^2 S L).  The five linears are gcgcn_gemm calls made by the caller (gcgcn_b200/edgefeat.py); the entry
 * points below are the rest.  Tables are built on the host from the wire format (edgefeat.EdgeTables):
 *   active tokens a: tokens [0, Lact) of every document that has an active slot, documents back to back;
 *   active slots s (sorted by document, then pair): sentence tokens [0, slot_len), mention spans, node rows;
 *   active pairs p: global pair index, CSR over their slots, denominator float32(sent_num) + 1e-10 (G:206, 213).   */
typedef struct gcgcn_edge_tables {
    int32_t num_tokens;           /* active tokens                                                         */
    int32_t num_slots;            /* active slots                                                          */
    int32_t num_pairs;            /* active pairs                                                          */
    int32_t att_total;            /* attention entries: sum over slots of 2 * slot_len                     */
    int32_t dis_plus;             /* config/Config.py:119                                                  */
    int32_t reserved;
    const int32_t* tok_first;     /* [num_tokens] active-token index of token 0 of the same document       */
    const int32_t* tok_slot_lo;   /* [num_tokens] first active slot of the token's document                */
    const int32_t* tok_slot_hi;   /* [num_tokens] one past the last                                        */
    const int32_t* slot_tok0;     /* [num_slots] active-token index of the document's token 0              */
    const int32_t* slot_len;      /* [num_slots] min(sentence end, document length)                        */
    const int32_t* slot_span;     /* [num_slots][4] head mention [h0, h1], tail mention [t0, t1] (C:187-201) */
    const int32_t* slot_att;      /* [num_slots] offset of the slot's 2 * slot_len attention entries       */
    const int32_t* slot_rowi;     /* [num_slots] node row of the pair's row entity i                       */
    const int32_t* slot_rowj;     /* [num_slots] node row of its column entity j                           */
    const int64_t* pair_idx;      /* [num_pairs] global pair index (pair_ptr[b] + i * n + j)               */
    const int32_t* pair_slot_ptr; /* [num_pairs + 1]                                                       */
    const float* pair_denom;      /* [num_pairs]                                                           */
    const int32_t* node_ctr_ptr;  /* [total_nodes + 1] CSR: (slot * 2 + side) entries embedding this node row */
    const int32_t* node_ctr;
    /* optional (may be 0 / NULL): the documents that have active slots, for the one-CTA-per-document word kernels   */
    int32_t num_active_docs;
    int32_t max_active_len;       /* longest run of active tokens of one document                              */
    const int32_t* adoc_tok0;     /* [num_active_docs] active-token index of the document's token 0            */
    const int32_t* adoc_len;      /* [num_active_docs] its active tokens                                       */
    const int32_t* adoc_slot_lo;  /* [num_active_docs] its active slots [lo, hi)                               */
    const int32_t* adoc_slot_hi;
} gcgcn_edge_tables;
/* scratch any entry point below needs */
size_t gcgcn_edgefeat_ws_bytes(int32_t num_tokens, int32_t att_total, int32_t num_slots, int32_t num_pairs,
                               int64_t total_pairs);
/* T[a][k] = wa . tanh(SF[a] + DF[k]) + ba;  SF [tokens,128], DF [21,128], T [tokens,21]                    */
int gcgcn_word_table_fwd(const float* SF, const float* DF, const float* wa, const float* ba, int32_t tokens, float* T,
                         void* stream);
/* dparams [21*128 + 128 + 4] = dDF, dwa, dba, 3 floats of padding                                          */
int gcgcn_word_table_bwd(const float* SF, const float* DF, const float* wa, const float* dT, int32_t tokens, float* dSF,
                         float* dparams, void* ws, size_t ws_bytes, void* stream);
/* per (slot, side): att = softmax over the sentence tokens of T[l][pos(l)] (G:186-187; the -1e5 fill of the tokens
 * outside the sentence underflows to exactly 0), cwa[slot][side*128 ..] = sum_l att[l] ctx[l] (G:188).
 * ctx [tokens,128] = the active rows of context_output; att [att_total] is an output saved for backward.     */
int gcgcn_word_pool_fwd(const gcgcn_edge_tables* tabs, const float* T, const float* ctx, float* att, float* cwa,
                        void* stream);
int gcgcn_word_pool_bwd(const gcgcn_edge_tables* tabs, const float* ctx, const float* att, const float* dcwa,
                        float* dctx, float* dT, void* ws, size_t ws_bytes, void* stream);
/* per active pair: score_side[s] = va . tanh(sfeat[s] + nfeat[j | i]) + ca (G:202-204; side h embeds the column
 * entity, side t the row entity, G:320-321), csa_side = sum_s relu(score_side[s]) cw[s] / denom (G:212-213).
 * score [slots,2] is saved for backward; csa [pairs,256] = (h | t).                                          */
int gcgcn_sent_pool_fwd(const gcgcn_edge_tables* tabs, const float* cw, const float* sfeat, const float* nfeat,
                        const float* va, const float* ca, float* score, float* csa, void* stream);
/* dparams [128 + 4] = dva, dca, 3 floats of padding                                                        */
int gcgcn_sent_pool_bwd(const gcgcn_edge_tables* tabs, int32_t total_nodes, const float* cw, const float* sfeat,
                        const float* nfeat, const float* va, const float* score, const float* dcsa, float* dcw,
                        float* dsfeat, float* dnfeat, float* dparams, void* ws, size_t ws_bytes, void* stream);
/* e[p] = bias for every pair, bias + rows[k] for the active pair pair_idx[k] (rows = csa W_ls^T, no bias).
 * bwd: drows[k] = de[pair_idx[k]], dbias = column sums of de over ALL pairs.                                */
int gcgcn_edge_fill_fwd(const float* bias, const float* rows, const int64_t* pair_idx, int32_t num_pairs,
                        int64_t total_pairs, int32_t edge_dtype, void* e, void* stream);
int gcgcn_edge_fill_bwd(const void* de, const int64_t* pair_idx, int32_t num_pairs, int64_t total_pairs,
                        int32_t edge_dtype, float* drows, float* dbias, void* ws, size_t ws_bytes, void* stream);
/* out[c] = sum_r X[r][c] (bias gradients of the linears); ws >= gcgcn_edgefeat_ws_bytes(...) or 4 MB         */
int gcgcn_colsum(const float* X, int32_t M, int32_t N, int32_t ldx, float* out, void* ws, size_t ws_bytes, void* stream);

/* ---- relation classifier and loss (SURVEY.md 8f row 2, second half) -------------------------------------------
 * logits = bili_layer_01(h, t) + classification_layer_01(cat[h, t])  (G:356-358) with h, t = entity_feature_h / _t
 * [total_pairs, 128] from gcgcn_pair_dense_fwd.  The bilinear form runs on gcgcn_gemm as Y = h W' (W' = the
 * [R, 128, 128] weight viewed as [128, R*128], 3xTF32 tcgen05 tiles) followed by the reductions below; the caller
 * (gcgcn_b200/classifier.py) walks the pairs in chunks so that Y stays within a fixed workspace.
 *   reduce: out[p][r] (+)= sum_b Y[p][r*128 + b] t[p][b] (+ bias[r])        Y [rows, R*128], out row stride ldo
 *   outer:  dY[p][r*128 + b] = dout[p][r] t[p][b]                            (then dh = dY W'^T, dW' = h^T dY)
 *   dt:     dt[p][b] = sum_r dout[p][r] Y[p][r*128 + b]                                                        */
/* Fused forward: out[p][r] (+)= sum_{a,b} h[p][a] W'[a][r*128 + b] t[p][b] + bias[r] in ONE tensor-core pass -- h stays
 * resident in tensor memory per 128-pair tile, W' streams through shared memory as pre-split blobs, and the epilogue
 * contracts every 128 x 128 accumulator tile (one relation) with t straight out of TMEM, so h W' never exists.
 * Wm = W' [128, relations*128] row-major; ws >= gcgcn_bilinear_ws_bytes(rows, relations).                       */
size_t gcgcn_bilinear_ws_bytes(int32_t rows, int32_t relations);
int gcgcn_bilinear_fwd(const float* h, const float* t, const float* Wm, const float* bias, int32_t rows,
                       int32_t relations, int32_t accumulate, float* out, int32_t ldo, void* ws, size_t ws_bytes,
                       void* stream);
/* Fused backward of the bilinear form for rows >= 8192 (GCGCN_ERR_UNSUPPORTED below that: use the three kernels
 * further down), no [rows, relations*128] intermediate:
 *   dt[p][b] = sum_r dout[p][r] (h W')[p][r*128 + b]      row-accumulate epilogue on the TMEM-resident GEMM, A = h, B = Wm
 *   dh[p][a] = sum_r dout[p][r] (t W'')[p][r*128 + a]     the same with A = t, B = Wm2 (W viewed as [128 (b), relations*128 (r, a)])
 *   dWm[a][r*128 + b] = beta dWm + sum_p h[p][a] dout[p][r] t[p][b]   weight-gradient GEMM whose [rows, relations*128]
 *                       operand is generated in the producers from t and dout (never stored)
 * dout [rows, relations] row-major.  ws >= gcgcn_bilinear_bwd_ws_bytes(rows, relations).                          */
size_t gcgcn_bilinear_bwd_ws_bytes(int32_t rows, int32_t relations);
int gcgcn_bilinear_bwd(const float* h, const float* t, const float* Wm, const float* Wm2, const float* dout, int32_t rows,
                       int32_t relations, float beta, float* dh, float* dt, float* dWm, void* ws, size_t ws_bytes,
                       void* stream);
int gcgcn_bilinear_reduce_fwd(const float* Y, const float* t, const float* bias, int32_t rows, int32_t relations,
                              int32_t accumulate, float* out, int32_t ldo, void* stream);
int gcgcn_bilinear_outer_bwd(const float* dout, int32_t ldd, const float* t, int32_t rows, int32_t relations, float* dY,
                             void* stream);
int gcgcn_bilinear_dt_bwd(const float* dout, int32_t ldd, const float* Y, int32_t rows, int32_t relations, float* dt,
                          void* stream);
/* cls_feature of the BERT variant (models/GraphCNN_multihead_bert_gate_cls.py:346-347): a per-document vector
 * v[b] = linear_cls(cls_feat_b) added to the logits of every pair of document b.  z [total_pairs, relations] in place;
 * bwd: dv[b] = sum of dz over the document's pairs.                                                              */
int gcgcn_doc_bias_fwd(const gcgcn_batch* bt, const float* v, int32_t relations, float* z, void* stream);
int gcgcn_doc_bias_bwd(const gcgcn_batch* bt, const float* dz, int32_t relations, float* dv, void* stream);
/* The trainer's loss, config/Config.py:355-364, per document of the batch: predict = sigmoid(logits) (C:355), then the
 * mean over the ordered pairs i != j of BCELoss(predict[i][j], label[i][j]) (mean over the R relation slots, C:361-364;
 * torch's clamping of the logs at -100 included).  logits, labels [total_pairs, R]; loss [num_docs].
 * bwd: dlogits = d(sum_b dloss[b] loss[b]) / dlogits (zero on the diagonal pairs).                              */
int gcgcn_pair_bce_fwd(const gcgcn_batch* bt, const float* logits, const float* labels, int32_t relations, float* loss,
                       void* stream);
int gcgcn_pair_bce_bwd(const gcgcn_batch* bt, const float* logits, const float* labels, int32_t relations,
                       const float* dloss, float* dlogits, void* stream);

/* ---- relation evaluation (config/Config.py:432-561; Ign F1 of config/Config_bert.py:626-650) ---------------------
 * The DocRED baseline evaluation on the device.  A candidate is (document, row i, column j, relation r) with i != j and
 * 1 <= r < R; its id is its position in insertion order (batches in call order, then documents, i, j, r ascending).
 * Global ids (gcgcn_rank_candidates_at) number the candidates of a whole evaluated set of G documents instead: document
 * g's first id is sum_{g' < g} (n_g'^2 - n_g')(R - 1), and inside a document the order is i, j, r as above.  A set
 * evaluated in shards (one per GPU) then ranks each shard with gcgcn_rank_sort and merges the sorted runs with
 * gcgcn_rank_merge; the merged ranking equals the ranking of the whole set.
 *   score   = 1 / (1 + exp(-logit))                float32, the loss kernel's sigmoid
 *   correct = labels[p][r] > 0.5;  intrain = intrain[p][r] != 0 (counts only where correct)
 * Ranking: score descending, stable (equal scores keep id order).  At ranked position k (0-based), with c_k / t_k the
 * running counts of correct / correct-and-intrain candidates and T = total_recall:
 *   x_k = f32(c_k / T), y_k = f32(c_k / (k + 1))   (double division, one rounding)
 *   f1_k = (2 x_k y_k) / ((x_k + y_k) + 1e-20)       (float32, every operation rounded, no contraction)
 *   yi_k = 0 if t_k == c_k, else f32((c_k - t_k) / (k + 1 - t_k))   (Ign precision; the x axis stays x_k)
 *   best_pos = first argmax of f1_k, theta = its score, auc = sum_k f32((x_{k+1} - x_k) (y_{k+1} + y_k) / 2) (terms as
 *   np.trapezoid forms them in float32, summed in float64 in a fixed order; 0 for one candidate)
 *   w = best_pos if input_theta == -1, else the last position whose score > input_theta (0 if none).
 * One evaluator holds fewer than 2^30 candidates (the payload packs id << 2 | intrain << 1 | correct):
 * GCGCN_ERR_UNSUPPORTED beyond that; with global ids the whole set's candidates count.  Every result is
 * bit-reproducible.                                                                                                */
#define GCGCN_RANK_TILE 4096          /* candidates per CTA of the sort and curve kernels */
#define GCGCN_RANK_MAX_CANDIDATES (1LL << 30)

typedef struct gcgcn_rank_result {    /* 80 bytes, written on the device by gcgcn_rank_curve                */
    int64_t count;                    /*  0: candidates N                                                 */
    int64_t total_recall;             /*  8: T actually used (>= 1)                                       */
    int64_t best_pos;                 /* 16: first argmax of f1_k                                         */
    int64_t w;                        /* 24: position the *_at_w fields are read at                       */
    double auc;                       /* 32                                                               */
    double ign_auc;                   /* 40: 0 without intrain                                            */
    float f1;                         /* 48: f1_k at best_pos                                             */
    float theta;                      /* 52: score at best_pos                                            */
    float f1_at_w;                    /* 56                                                               */
    float precision_at_w;             /* 60: y_w                                                          */
    float recall_at_w;                /* 64: x_w                                                          */
    float ign_f1;                     /* 68: max_k of the Ign f1 (0 without intrain)                      */
    float ign_f1_at_w;                /* 72: (0 without intrain)                                          */
    float reserved;                   /* 76                                                               */
} gcgcn_rank_result;

/* workspace of gcgcn_rank_sort and gcgcn_rank_curve for `count` candidates (about 8 bytes per candidate; any
 * alignment: the library aligns inside it)                                                                         */
size_t gcgcn_rank_ws_bytes(int64_t count);
/* Scores and payloads of every candidate of one batch: logits / labels [total_pairs, relations] float32, intrain
 * [total_pairs, relations] uint8.  labels NULL: nothing is correct (unlabeled sets); intrain NULL: nothing is.
 * Candidate ids start at base_id (the count of earlier batches); score / payload receive this batch's
 * (total_pairs - total_nodes) (relations - 1) candidates at [id - base_id].  counters[0] += correct candidates,
 * counters[1] += NaN scores (int64, accumulated across batches).                                                    */
int gcgcn_rank_candidates(const gcgcn_batch* bt, const float* logits, int32_t relations, const float* labels,
                          const uint8_t* intrain, int64_t base_id, float* score, uint32_t* payload, int64_t* counters,
                          void* stream);
/* The same with global ids: doc_base [num_docs] int64 (device) is the first global id of each document of the batch.
 * score / payload receive the batch's candidates compactly from position 0, exactly as gcgcn_rank_candidates with
 * base_id 0 would; only the id packed in the payload differs.  The caller keeps every id below 2^30.              */
int gcgcn_rank_candidates_at(const gcgcn_batch* bt, const float* logits, int32_t relations, const float* labels,
                             const uint8_t* intrain, const int64_t* doc_base, float* score, uint32_t* payload,
                             int64_t* counters, void* stream);
/* Stable ranking of `count` candidates: sorted_key[k] = ~bits(score) of the k-th ranked candidate (ascending keys =
 * descending scores), sorted_payload[k] its payload.  ws >= gcgcn_rank_ws_bytes(count).                           */
int gcgcn_rank_sort(const float* score, const uint32_t* payload, int64_t count, uint32_t* sorted_key,
                    uint32_t* sorted_payload, void* ws, size_t ws_bytes, void* stream);
/* The curve over a ranking from gcgcn_rank_sort; writes *result (device memory) on the stream.  total_recall < 1
 * means 1.  has_intrain = 0 leaves the Ign fields 0.  The result is meaningless if any score is NaN.
 * sorted_payload 16-byte aligned.                                                                               */
int gcgcn_rank_curve(const uint32_t* sorted_key, const uint32_t* sorted_payload, int64_t count, int64_t total_recall,
                     int32_t has_intrain, double input_theta, gcgcn_rank_result* result, void* ws, size_t ws_bytes,
                     void* stream);
/* Workspace of gcgcn_rank_merge for na + nb = count outputs (8 bytes per 4096 outputs; any alignment).          */
size_t gcgcn_rank_merge_ws_bytes(int64_t count);
/* Merge two rankings, each ascending by (key, payload) read as one 64-bit value (key high): the output, na + nb long,
 * ascends the same way; on an exact duplicate the item of A comes first.  Rankings of disjoint candidate sets with
 * distinct (global) ids merge into the ranking of their union.  Deterministic, no atomics; na or nb may be 0.
 * Outputs 16-byte aligned and disjoint from the inputs; na + nb < 2^30.  Moves 16 bytes per output.             */
int gcgcn_rank_merge(const uint32_t* key_a, const uint32_t* payload_a, int64_t na, const uint32_t* key_b,
                     const uint32_t* payload_b, int64_t nb, uint32_t* key_out, uint32_t* payload_out, void* ws,
                     size_t ws_bytes, void* stream);
/* The curve's points at every ranked position k (the reference's pr_x, pr_y and the Ign pr_y): x[k] = x_k,
 * y[k] = y_k, y_ign[k] = yi_k (written only if has_intrain), float32 [count].  total_recall < 1 means 1;
 * ws >= gcgcn_rank_ws_bytes(count); sorted_payload 16-byte aligned.                                              */
int gcgcn_rank_curve_points(const uint32_t* sorted_payload, int64_t count, int64_t total_recall, int32_t has_intrain,
                            float* x, float* y, float* y_ign, void* ws, size_t ws_bytes, void* stream);
/* The first `rows` ranked candidates (rows <= count, the ranking's length) as (doc, row, col, relation, score) int32 /
 * float32 [rows].  doc_offsets
 * [num_docs + 1] int64: first candidate id of each document, (n_b^2 - n_b)(relations - 1) apart; doc_n [num_docs]
 * int32 entity counts.  doc is the document's index in doc_offsets.                                               */
int gcgcn_rank_decode(const uint32_t* sorted_key, const uint32_t* sorted_payload, int64_t rows, int64_t count,
                      const int64_t* doc_offsets, const int32_t* doc_n, int32_t num_docs, int32_t relations, int32_t* doc,
                      int32_t* row, int32_t* col, int32_t* relation, float* score, void* stream);

/* ---- relation evaluation per relation -----------------------------------------------------------------------------
 * A candidate's relation is (id mod (R - 1)) + 1 (every document's first id is a multiple of R - 1, for local and
 * global ids), and each relation holds exactly count / (R - 1) of the candidates of a ranking.
 * Per-relation result: entry r - 1 is what gcgcn_rank_curve returns when given only relation r's candidates, in their
 * order in the ranking (which, the ranking being stable, is the stable ranking of those candidates alone); every field
 * keeps its meaning with positions counted inside the relation's own ranking.  T_r = total_recall[r - 1], or else the
 * number of correct candidates of r; < 1 means 1.  input_theta[r - 1] = -1 selects the relation's best-F1 position;
 * any other value the last position whose score > input_theta[r - 1], or 0 if there is none.
 * Selection at per-relation thresholds: every candidate whose score > theta[relation - 1], in ranked order.  With m
 * candidates selected, c of them correct and t correct and intrain, and T the total recall: precision =
 * f32(c / m) (0 when m = 0), recall = f32(c / T), f1 = (2 recall precision) / ((recall + precision) + 1e-20) and Ign
 * f1 the same with the Ign precision of (c, t, m) (the roundings of the curve above).
 * At most 256 relations r >= 1 (R <= 257: one 8-bit digit).  Every entry point is deterministic and bit-reproducible,
 * writes only the caller's memory and enqueues on the stream.                                                       */
/* workspace of gcgcn_rank_by_relation, gcgcn_rank_curve_relations and gcgcn_rank_select (any alignment)            */
size_t gcgcn_rank_relations_ws_bytes(int64_t count, int32_t relations);
/* Stable partition of a ranking (gcgcn_rank_sort / gcgcn_rank_merge) by relation: relation r's candidates, in ranked
 * order, at [(r - 1) count / (R - 1), r count / (R - 1)).  count % (R - 1) != 0: GCGCN_ERR_INVALID_ARG; R - 1 > 256:
 * GCGCN_ERR_UNSUPPORTED.  Outputs disjoint from the inputs.  Moves 20 bytes per candidate.                         */
int gcgcn_rank_by_relation(const uint32_t* sorted_key, const uint32_t* sorted_payload, int64_t count, int32_t relations,
                           uint32_t* rel_key, uint32_t* rel_payload, void* ws, size_t ws_bytes, void* stream);
/* The per-relation results over a partition from gcgcn_rank_by_relation: results [R - 1] (device memory).
 * total_recall [R - 1] int64 (device) or NULL; input_theta [R - 1] double (device).  rel_payload 16-byte aligned.  */
int gcgcn_rank_curve_relations(const uint32_t* rel_key, const uint32_t* rel_payload, int64_t count, int32_t relations,
                               const int64_t* total_recall, int32_t has_intrain, const double* input_theta,
                               gcgcn_rank_result* results, void* ws, size_t ws_bytes, void* stream);
/* Selection of a ranking at theta [R - 1] float32 (device): out_key / out_payload [count] receive the selected
 * candidates, in ranked order, from position 0 (gcgcn_rank_decode lists them); counts [3] int64 (device) = m, c, t.
 * Inputs 16-byte aligned; outputs disjoint from them.                                                               */
int gcgcn_rank_select(const uint32_t* sorted_key, const uint32_t* sorted_payload, int64_t count, int32_t relations,
                      const float* theta, uint32_t* out_key, uint32_t* out_payload, int64_t* counts, void* ws,
                      size_t ws_bytes, void* stream);

/* ---- training step of config 5 (new work: the reference has no multi-GPU path, SURVEY.md 8e) ----
 * Fused Adam over ONE flat float32 buffer holding every hot-path parameter, with the semantics of
 * torch.optim.Adam as the reference's trainer constructs it (config/Config.py:300: lr only, betas
 * (0.9, 0.999), eps 1e-8, weight_decay 0).  `grads` is the (all-reduced) flat gradient bucket,
 * grad_scale is folded in (1/world_size or 1/documents), `step` counts from 1.  In place on
 * params / exp_avg / exp_avg_sq; all four buffers 16-byte aligned.                              */
int gcgcn_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t count,
                    float lr, float beta1, float beta2, float eps, float weight_decay, float grad_scale,
                    int32_t step, void* stream);

/* ---- dense projection used by the entry points above (exported for tests) ----------------
 * C = alpha * op(A) op(B) + beta * C (+ bias broadcast over rows), row-major float32.
 * trans_a / trans_b: 0 = as stored, 1 = transposed.  K may be huge (weight gradients reduce
 * over every node row of the batch); the split-K partials live in ws.                      */
int gcgcn_gemm(int32_t trans_a, int32_t trans_b, int32_t M, int32_t N, int32_t K, float alpha,
               const float* A, int32_t lda, const float* B, int32_t ldb, float beta, float* C,
               int32_t ldc, const float* bias, void* ws, size_t ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GCGCN_B200_H */
