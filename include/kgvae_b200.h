/*
 * kgvae_b200.h - C ABI of the B200-native GCN-VAE link-prediction hot path.
 *
 * The reference (karenyang/GCN-VAE) has no FFI layer: its hot path sits behind Python
 * module calls into PyTorch/DGL.  Each entry point below replaces one of those calls;
 * the "replaces" line cites the reference interface (file:line under /root/reference).
 * The Python host side (gcn-vae_b200/ops.py) binds these with ctypes; see INTEGRATION.md.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch caching allocator);
 *     nothing is allocated or freed across this boundary; workspaces are caller-provided
 *   - `stream` is the caller's cudaStream_t (as void*); all work is stream-ordered
 *   - indices are int32, features fp32, row-major, contiguous unless a leading dimension
 *     is passed
 *   - return value: 0 on success, negative on error; kg_last_error() gives the message
 *     (thread-local); no C++ exception crosses the boundary
 */
#ifndef KGVAE_B200_H_
#define KGVAE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KG_OK 0
#define KG_ERR_INVALID -1
#define KG_ERR_CUDA -2
#define KG_ERR_WORKSPACE -3

const char* kg_last_error(void);
int kg_version(void);
/* device attributes used for grid sizing (SM count etc.); also a liveness check */
int kg_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* Peer-visible buffers for destination-partitioned training (new; the reference is single-process):
 * cudaMalloc'ed, zero-filled memory exported with CUDA IPC (64-byte handle) and opened by the other
 * ranks of the node on their own current device with lazy peer access; the returned pointers go
 * into the x_parts table of kg_bdd_rel_fwd / kg_bdd_rel_bwd. */
int kg_peer_alloc(size_t bytes, void** ptr, unsigned char* handle_out /* 64 bytes */);
int kg_peer_open(const unsigned char* handle /* 64 bytes */, void** ptr);
int kg_peer_close(void* ptr);
int kg_peer_free(void* ptr);

/* ------------------------------------------------------------------------------------
 * a1  graph construction
 * replaces: utils.build_graph_from_triplets / comp_deg_norm  kgvae/utils.py:127-150
 *           node_norm_to_edge_norm                           kgvae/link_predict.py:95-100
 * Input: T triplets (src, rel, dst).  Output: 2T directed edges (reverse edges carry
 * rel + num_rels) in ascending (dst, src, rel) order - the reference's
 * sorted(zip(dst, src, rel)) - plus everything the kernels need:
 *   e_src/e_dst/e_type [2T], row_ptr [N+1] (dst-CSR), node_norm [N] = 1/in_deg (0 if 0),
 *   fwd_pack [2T] int4 {src, etype, bits(norm[dst]), dst}        (dst-major order)
 *   col_ptr [N+1], bwd_pack [2T] int4 {dst, etype, bits(norm), edge_id}  (src-major order)
 *   rel_ptr [2R+1], rel_pack [2T] int4 {src, dst, etype, bits(norm)}     (etype-major)
 * fwd_pack and bwd_pack are optional (NULL: that ordering is not built; the bdd message passing
 * only walks rel_pack).  Limits: N < 2^24, 2R < 2^16.
 * ---------------------------------------------------------------------------------- */
size_t kg_graph_build_workspace_bytes(int n_triplets);
int kg_graph_build(const int32_t* src, const int32_t* rel, const int32_t* dst, int n_triplets,
                   int num_nodes, int num_rels,
                   int32_t* e_src, int32_t* e_dst, int32_t* e_type,
                   int32_t* row_ptr, float* node_norm,
                   void* fwd_pack, int32_t* col_ptr, void* bwd_pack,
                   int32_t* rel_ptr, void* rel_pack,
                   void* workspace, size_t workspace_bytes, void* stream);

/* Relabelling of B sampled triples for a subgraph padded to a fixed node budget (kgvae/utils.py:85-124,
 * np.unique((src, dst), return_inverse=True)), with every size fixed by B and cap - no host read-back, so the call
 * can be captured in a CUDA graph.  picked [B, 3] int32 (s, r, o).  Outputs:
 *   node_id [cap]: the n_valid distinct entity ids in ascending order, then padding rows i = n_valid .. cap-1
 *                  holding entity i (in range; no id occurs more than twice)
 *   src / dst [B]: relabelled end-points (0 .. n_valid-1), rel [B]: the relation column, n_valid [1]: device int.
 * Needs 0 < cap <= min(2B, num_nodes) and cap >= the number of distinct ids (entity ids < num_nodes); with fewer
 * rows than distinct ids, n_valid is clamped to cap and the ids past it are dropped. */
size_t kg_sample_relabel_workspace_bytes(int n_picks);
int kg_sample_relabel(const int32_t* picked, int n_picks, int num_nodes, int cap, int32_t* node_id,
                      int32_t* src, int32_t* rel, int32_t* dst, int32_t* n_valid,
                      void* workspace, size_t workspace_bytes, void* stream);

/* Neighbourhood-expansion edge sampler (new device form of utils.sample_edge_neighborhood, kgvae/utils.py:33-76):
 * one launch draws n_samples independent samples of sample_size distinct triples, one warp per sample.  Each pick
 * consumes KG_NEIGHBOR_WORDS caller words: word 0 draws the vertex (~ cnt * seen, or ~ [cnt > 0] when that sums to
 * 0), words 1..KG_NEIGHBOR_TRIES are the reference's rejection tries on its adjacency list, the next word picks
 * among its unpicked entries when every try hit a picked edge.  tests/neighbor_mirror.py is the specification; the
 * output depends only on the graph and the words.
 *   adj_ptr [N+1], adj [2T][2] (edge id, other end): per entity, ascending edge id, the subject end first for a
 *                  self-loop (utils.get_adj_and_degrees)
 *   words [n_samples, sample_size, KG_NEIGHBOR_WORDS] uniform 32-bit, picks [n_samples, sample_size] edge ids,
 *   fallbacks [n_samples] (or NULL): picks that needed the unpicked-entry scan
 * The per-sample state lives in shared memory when it fits, else in the workspace (one slab per resident warp).
 * kg_neighbor_sample_plan gives the samples resident in one wave (bounded by a 1 GiB budget for words, picks and
 * slabs) and the workspace bytes for that many.  Needs 1 <= sample_size <= T and 0 < N, T < 2^30. */
#define KG_NEIGHBOR_WORDS 8
#define KG_NEIGHBOR_TRIES 6
int kg_neighbor_sample_plan(int num_nodes, int n_triples, int sample_size, int* samples_per_launch,
                            size_t* workspace_bytes);
int kg_neighbor_sample(const int32_t* adj_ptr, const int32_t* adj, int num_nodes, int n_triples, int sample_size,
                       int n_samples, const uint32_t* words, int32_t* picks, int32_t* fallbacks,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Same index structures from an edge list the caller already ordered (the DGLGraph
 * surface: g.add_edges(src, dst) + etypes + per-edge norm, kgvae/utils.py:141-148).
 * Edges need not be sorted; the original edge order is kept as the tie-break so the
 * per-destination summation order equals the reference's edge order. */
size_t kg_graph_index_workspace_bytes(int n_edges);
int kg_graph_index(const int32_t* e_src, const int32_t* e_dst, const int32_t* e_type,
                   const float* e_norm /* [E] or NULL (=1) */, int n_edges, int num_nodes,
                   int num_etypes,
                   int32_t* row_ptr, void* fwd_pack, int32_t* col_ptr, void* bwd_pack,
                   int32_t* rel_ptr, void* rel_pack,
                   void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * a2  embedding lookup
 * replaces: EmbeddingLayer.forward   kgvae/model.py:185-191
 * ---------------------------------------------------------------------------------- */
int kg_embedding_fwd(const float* table, const int32_t* ids, int n, int dim, float* out, void* stream);
/* grad_table must be zero-filled by the caller; rows are accumulated (duplicates allowed) */
int kg_embedding_bwd(const float* grad_out, const int32_t* ids, int n, int dim, float* grad_table,
                     void* stream);

/* ------------------------------------------------------------------------------------
 * a3  RelGraphConv, regularizer="bdd" (block-diagonal decomposition)
 * replaces: dgl.nn.pytorch.RelGraphConv.forward(g, x, etypes, norm), constructed at
 *           kgvae/model.py:54-59, called at kgvae/model.py:110-111
 * weight [R, B*si*so] row-major (b, i, o) as in DGL.
 * ---------------------------------------------------------------------------------- */
/* derived layouts, rebuilt whenever `weight` changes:
 *   w_fwd [R, si, B*so]: w_fwd[r][i][b*so+o] = weight[r][b][i][o]
 *   w_bwd [R, so, B*si]: w_bwd[r][o][b*si+i] = weight[r][b][i][o]                     */
int kg_bdd_weight_layouts(const float* weight, int num_etypes, int num_bases, int si, int so,
                          float* w_fwd, float* w_bwd, void* stream);
/* Message passing (rgcn_bdd_rel.cu): edges walked in relation-major order - rel_pack from
 * kg_graph_index, or a node-tiled list from kg_graph_rel_tiled - so that a thread keeps its columns
 * of the relation's block weights in registers for a run of edges; messages are accumulated with
 * vector reductions.  agg / dx / dweight must be zero-filled by the caller; dx may be NULL.
 *   fwd:  agg[dst] += norm * blockdiag(W[etype]) x[src]
 *   bwd:  dx[src] += norm * blockdiag(W[etype])^T dagg[dst];  dweight[etype] += norm * x[src] (x) dagg[dst]
 * hints: KG_HINT_STREAM_X / KG_HINT_STREAM_D mark the gathered matrix (x / dagg) as streamed from
 * HBM (evict-first in L2) so that it does not displace the L2-resident tile being reduced into. */
#define KG_HINT_STREAM_X 1
#define KG_HINT_STREAM_D 2
#define KG_HINT_TILE_RESIDENT 4   /* node-tiled list: keep the rows reduced into (and x in backward) evict-last */
/* x_parts (optional, device array of pointers) + part_rows: destination-partitioned training - source
 * rows live in one block per rank (row r = row r % part_rows of x_parts[r / part_rows], peer blocks
 * mapped with CUDA IPC) and are fetched over NVLink by the kernel's own gather stage, replacing the
 * all-gather of layer inputs (5x5 / 5x10 block shapes only; pass NULL, 0 and x otherwise). */
int kg_bdd_rel_fwd(const float* x, const void* x_parts, int part_rows, const void* rel_pack, int n_edges,
                   const float* weight, const float* w_fwd, int num_bases, int si, int so, float* agg,
                   int hints, void* stream);
int kg_bdd_rel_bwd(const float* x, const void* x_parts, int part_rows, const float* dagg,
                   const void* rel_pack, int n_edges, const float* weight, const float* w_bwd,
                   int num_bases, int si, int so, float* dx, float* dweight, int hints, void* stream);

/* Column chunks of the same layer (new; destination-partitioned training): blocks [block0, block0 + num_bases) of
 * num_bases_total only touch columns [block0 si, ...) of x and [block0 so, ...) of agg, so a chunk can run as
 * soon as ITS columns of the all-gathered layer input have arrived, and its source gradients can be
 * reduce-scattered while the next chunk computes.  x_chunk / dx_chunk: compact [n_src, num_bases si] matrices;
 * weight / dweight / agg / dagg: the full tensors.  5x5 and 5x10 blocks. */
int kg_bdd_rel_fwd_cols(const float* x_chunk, const void* rel_pack, int n_edges, const float* weight,
                        int block0, int num_bases, int num_bases_total, int si, int so, float* agg,
                        int hints, void* stream);
int kg_bdd_rel_bwd_cols(const float* x_chunk, const float* dagg, const void* rel_pack, int n_edges,
                        const float* weight, int block0, int num_bases, int num_bases_total, int si, int so,
                        float* dx_chunk, float* dweight, int hints, void* stream);
/* The reference model's block shapes (5x5, 5x10; rgcn_bdd_own.cuh) read `weight` in the DGL layout
 * directly - a thread owns whole diagonal blocks in registers - and need no derived layout: pass
 * w_fwd / w_bwd = NULL when this returns 0.  Other shapes need kg_bdd_weight_layouts first. */
int kg_bdd_layouts_needed(int num_bases, int si, int so);

/* Node-tiled relation-major edge list for graphs whose feature matrices exceed L2 (wikikg2 / AM
 * shapes; new - the reference has no counterpart, DGL walks edges in insertion order):
 * records {src, dst, etype, bits(norm)} ordered by (tile(node), etype, original order) where
 * node = dst (by_src = 0, forward: the rows reduced into are agg[dst]) or src (by_src = 1,
 * backward: dx[src]) and tile(node) = node / tile_nodes.  One tile's rows stay L2-resident while
 * its edges are processed, so the per-edge HBM traffic is the gathered row only.
 * e_norm may be NULL (norm 1).  Limits: bits(num_nodes / tile_nodes) + bits(num_etypes) <= 32. */
size_t kg_graph_rel_tiled_workspace_bytes(int n_edges);
int kg_graph_rel_tiled(const int32_t* e_src, const int32_t* e_dst, const int32_t* e_type,
                       const float* e_norm, int n_edges, int num_nodes, int num_etypes,
                       int tile_nodes, int by_src, void* pack_out,
                       void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * a4  RelGraphConv, regularizer="basis" (entity classification)
 * replaces: dgl.nn.pytorch.RelGraphConv("basis").forward as constructed at
 *           kgvae/entity_classify.py:30-43 (W_r = sum_b w_comp[r,b] V_b; V [NB, in, out])
 * Integer node-id features (in = num_nodes): msg_e = norm_e * sum_b coef[r,b] V[b, id_e, :] without
 * ever forming the [R, in, out] table (coef NULL: NB == R and msg_e = norm_e * V[r, id_e, :]).
 * Dense features: msg_e = norm_e * x[src] @ W_r with W [R, in, out] composed by the caller (GEMM).
 * `out` must hold the self-loop term (or zeros) on entry; gradients are accumulated into
 * zero-filled buffers.  ids: optional int32 [n_src] row map (the 1-D feature tensor), NULL = identity.
 * ---------------------------------------------------------------------------------- */
int kg_basis_id_fwd(const float* V, const float* coef, const int32_t* ids, const int32_t* row_ptr,
                    const void* fwd_pack, int n_dst, int n_in, int num_bases, int out_feat, float* out,
                    void* stream);
int kg_basis_id_bwd(const float* V, const float* coef, const int32_t* ids, const float* g,
                    const void* rel_pack, int n_edges, int n_in, int num_bases, int out_feat,
                    float* dV, float* dcoef, void* stream);
/* Source-tiled variants for the reference's featureless input layer (ids == arange(num_nodes),
 * kgvae/entity_classify.py:63) with a composed basis (coef != NULL): a CTA takes consecutive source
 * nodes, so V is read once in contiguous runs and dV is WRITTEN once without atomics or zero-fill;
 * col_ptr / bwd_pack are the src-major list of kg_graph_index ({dst, etype, bits(norm), edge}).
 * kg_basis_id_src_eligible: 1 when the shape is covered (num_bases <= 64, out_feat <= 16). */
int kg_basis_id_src_eligible(int num_rels, int num_bases, int out_feat);
int kg_basis_id_src_fwd(const float* V, const float* coef, const int32_t* col_ptr, const void* bwd_pack,
                        int n_src, int num_rels, int num_bases, int out_feat, float* out, void* stream);
int kg_basis_id_src_bwd(const float* V, const float* coef, const float* g, const int32_t* col_ptr,
                        const void* bwd_pack, int n_src, int num_rels, int num_bases, int out_feat,
                        float* dV, float* dcoef, void* stream);
int kg_basis_dense_fwd(const float* x, const void* rel_pack, int n_edges, const float* W, int num_rels,
                       int in_feat, int out_feat, float* out, void* stream);
int kg_basis_dense_bwd(const float* x, const float* g, const void* rel_pack, int n_edges, const float* W,
                       int num_rels, int in_feat, int out_feat, float* dx, float* dW, void* stream);

/* out = dropout(act(agg + bias + loop)) tail of RelGraphConv.forward; backward of the same.
 * act: 0 identity, 1 relu.  drop_mask: [n, dim] keep-mask already scaled by 1/(1-p), or NULL. */
int kg_act_dropout_bwd(const float* grad_out, const float* out, const float* drop_mask, int act,
                       long long numel, float* grad_pre, void* stream);
/* The same with the bias gradient fused in: colsum[c] = sum_r grad_pre[r, c] (the `h_bias` / MaskedLinear
 * bias gradients autograd derives for kgvae/model.py:54-59 and kgvae/flow_network.py:15); workspace as for
 * kg_colsum (used only on the unfused path: cols % 4 != 0 or unaligned tensors). */
int kg_act_dropout_bwd_colsum(const float* grad_out, const float* out, const float* drop_mask, int act,
                              int rows, int cols, float* grad_pre, float* colsum, void* workspace,
                              size_t workspace_bytes, void* stream);
/* column sums of a [rows, cols] matrix (h_bias / MaskedLinear bias gradients); deterministic.
 * workspace: kg_colsum_workspace_bytes(rows, cols) */
size_t kg_colsum_workspace_bytes(int rows, int cols);
int kg_colsum(const float* x, int rows, int cols, float* out, void* workspace, size_t workspace_bytes,
              void* stream);

/* ------------------------------------------------------------------------------------
 * dense fp32 GEMM with fused epilogue (self-loop x@loop_weight kgvae/model.py:55,58 via DGL;
 * MaskedLinear kgvae/flow_network.py:15 and its backward)
 *   C[M,N] = epilogue( op(A)[M,K] * op(B)[K,N] )
 *   A(m,k) = A[m*lda + k] if !trans_a else A[k*lda + m];  B(k,n) likewise with ldb.
 *   epilogue: v = acc (+ bias[n]) (+ addend[m*ldc+n]); if relu v = max(v,0);
 *             if mask v *= mask[m*ldc+n]; C = v   (accumulate: C += v)
 * Products with M, N >= 64, K >= 32 and M*N*K >= 2^22 run on the tensor cores (tcgen05,
 * two-term fp16 split of both operands made inside the call, fp32 accumulate: fp32-accurate); they need
 * kg_gemm_f32_workspace_bytes(M, N, K) bytes of workspace (0 for the small-product FMA kernel).
 * ---------------------------------------------------------------------------------- */
size_t kg_gemm_f32_workspace_bytes(int M, int N, int K);
int kg_gemm_f32(const float* A, int lda, int trans_a, const float* B, int ldb, int trans_b,
                float* C, int ldc, int M, int N, int K,
                const float* bias, const float* addend, int relu, const float* mask,
                int accumulate, void* workspace, size_t workspace_bytes, void* stream);

/* Prepared operands of the tensor-core GEMM (new; the reference's torch.matmul has no counterpart).
 * kg_gemm_prepare splits a row-major fp32 matrix src[rows, cols] (row pitch ld) once into the two-term fp16
 * form the tensor-core product reads, under one power-of-two scale for the whole matrix, into a caller-owned
 * buffer of kg_gemm_prep_bytes(rows, cols) bytes (16-byte aligned).  The same prepared matrix serves every
 * product it takes part in, in either orientation: a layer prepares x, W and its upstream gradient g once for
 *   y = x W^T (kgvae/flow_network.py:15),  dx = g W,  dW = g^T x   (and likewise kgvae/model.py:55,58 via DGL).
 * kg_gemm_f32_prepared is kg_gemm_f32 on prepared operands: prep_a holds A as stored ([M, K], or [K, M] when
 * trans_a), prep_b holds B as stored ([K, N], or [N, K] when trans_b).  Only for products that
 * kg_gemm_f32_uses_tensor_cores(M, N, K); workspace kg_gemm_f32_prepared_workspace_bytes(M, N, K). */
int kg_gemm_f32_uses_tensor_cores(int M, int N, int K);
size_t kg_gemm_prep_bytes(int rows, int cols);
int kg_gemm_prepare(const float* src, int ld, int rows, int cols, void* prep, size_t prep_bytes, void* stream);
size_t kg_gemm_f32_prepared_workspace_bytes(int M, int N, int K);
int kg_gemm_f32_prepared(const void* prep_a, int trans_a, const void* prep_b, int trans_b,
                         float* C, int ldc, int M, int N, int K,
                         const float* bias, const float* addend, int relu, const float* mask,
                         int accumulate, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * a5  mean/variance heads + reparameterised sample
 * replaces: utils.gaussian_parameters kgvae/utils.py:323-339, utils.sample_gaussian :342-361
 * h2 [n, 2h] -> z_mean = h2[:, :h], z_var = softplus(h2[:, h:]) + 1e-8, z = m + eps*sqrt(v)
 * ---------------------------------------------------------------------------------- */
int kg_reparam_fwd(const float* h2, const float* eps, int n, int h, float* z_mean, float* z_var,
                   float* z, void* stream);
/* dh2 from (dz, dmean, dvar); any of dmean/dvar may be NULL */
int kg_reparam_bwd(const float* h2, const float* eps, const float* z_var, const float* dz,
                   const float* dmean, const float* dvar, int n, int h, float* dh2, void* stream);

/* ------------------------------------------------------------------------------------
 * a7  single-sample KL estimate against the mixture-of-Gaussians prior
 * replaces: KGVAE.get_kl kgvae/model.py:82-87 (log_normal :381-398, log_normal_mixture :364-378)
 * kl_rows[n] = logN(z_n; m_n, v_n) - log( (1/k) sum_i N(z_n; pm_i, pv_i) )   (flow term added
 * by the caller); resp [n, k] = posterior responsibilities saved for backward.
 * z_pre [2k, h]: rows 0..k-1 prior means, rows k..2k-1 raw variances (softplus + 1e-8).
 * prior_ws [3, k, h]: workspace written by fwd (variance, 1/(2 var), log sqrt var), read by bwd.
 * k <= 16.
 * ---------------------------------------------------------------------------------- */
int kg_kl_mog_fwd(const float* z, const float* z_mean, const float* z_var, const float* z_pre,
                  int n, int h, int k, float* prior_ws, float* kl_rows, float* resp, void* stream);
/* scale = dL/dkl / n.  dz_pre [2k, h] must be zero-filled by the caller. */
int kg_kl_mog_bwd(const float* z, const float* z_mean, const float* z_var, const float* z_pre,
                  const float* prior_ws, const float* resp, float scale, int n, int h, int k,
                  float* dz, float* dmean, float* dvar, float* dz_pre, void* stream);
/* kg_kl_mog_bwd with the rest of the loss head folded in (link_predict.py:74-91): one pass writes the TOTAL
 * gradient wrt z:  dz = coefs[0] scale dKL/dz + coefs[1] add + coefs[2] z  (add = dz of the DistMult + BCE
 * term, may be NULL; z = the regulariser's 2 z / (n h), the factor folded into coefs[2]); dmean, dvar, dz_pre
 * carry coefs[0] scale.  coefs: DEVICE [3], so the upstream gradient never visits the host. */
int kg_kl_mog_bwd_fused(const float* z, const float* z_mean, const float* z_var, const float* z_pre,
                        const float* prior_ws, const float* resp, float scale, int n, int h, int k,
                        const float* coefs, const float* add, float* dz, float* dmean, float* dvar,
                        float* dz_pre, void* stream);
/* The forward and the fused backward over the first n_valid (DEVICE int) of n_rows rows - a sampled subgraph padded
 * to a fixed node budget.  Valid rows compute exactly what kg_kl_mog_fwd / kg_kl_mog_bwd_fused compute on an
 * [n_valid, h] input (bitwise); padding rows get kl_rows = 0 (resp unwritten) and exact zeros in dz, dmean and
 * dvar, and add nothing to dz_pre.  The backward forms scale = 1 / n_valid itself. */
int kg_kl_mog_fwd_rows(const float* z, const float* z_mean, const float* z_var, const float* z_pre,
                       int n_rows, int h, int k, const int32_t* n_valid, float* prior_ws, float* kl_rows,
                       float* resp, void* stream);
int kg_kl_mog_bwd_fused_rows(const float* z, const float* z_mean, const float* z_var, const float* z_pre,
                             const float* prior_ws, const float* resp, int n_rows, int h, int k,
                             const int32_t* n_valid, const float* coefs, const float* add, float* dz,
                             float* dmean, float* dvar, float* dz_pre, void* stream);

/* ------------------------------------------------------------------------------------
 * a6  IAF: element update of one MADE pass
 * replaces: MADE.forward body kgvae/flow_network.py:91-96
 * net_out [n, 2d] = (mu | alpha).  col_mult [d] int32 = multiplicity of each column in the pass's
 * index list (flow_network.py:70-77,93): 0 keeps x_old[:, j]; otherwise
 * x_new[:, j] = z[:, j]*exp(alpha[:, j] + mu[:, j]) and the backward scales the column's gradient by
 * the multiplicity (autograd's index_put backward feeds every duplicate - the reference lists
 * column 0 twice in passes 2..n_hidden+2).
 * log_det[n] = sum_j alpha[n, j] (only written when log_det != NULL: the last pass).
 * ---------------------------------------------------------------------------------- */
int kg_iaf_update_fwd(const float* z, const float* net_out, const float* x_old,
                      const int32_t* col_mult, int n, int d, float* x_new, float* log_det,
                      void* stream);
int kg_iaf_update_bwd(const float* z, const float* net_out, const float* dx_new,
                      const float* dlog_det /* [n] or NULL */, const int32_t* col_mult, int n, int d,
                      float* dz, float* dnet_out, float* dx_old, void* stream);
/* column reversal (PermuteLayer kgvae/flow_network.py:28-30); its own inverse and backward */
int kg_reverse_columns(const float* x, int n, int d, float* out, void* stream);

/* ------------------------------------------------------------------------------------
 * a9  DistMult decoder + BCE-with-logits + L2 regulariser
 * replaces: LinkPredict.calc_score kgvae/link_predict.py:57-63, get_loss :71-78,
 *           regularization_loss :68-69
 * triplets [S, 3] int32 (s, r, o).  score_i = sum_d z[s,d] w[r,d] z[o,d] + shift
 * ---------------------------------------------------------------------------------- */
int kg_distmult_score(const float* z, const float* w, const int32_t* triplets, int n_triplets, int h,
                      const float* shift /* device scalar or NULL */, float* score, void* stream);
/* mean BCE-with-logits; also dscore_i = (sigmoid(score_i) - label_i) / S.
 * partial: workspace of kg_reduce_workspace_bytes(S) bytes; loss_out: 1 float */
size_t kg_reduce_workspace_bytes(long long n);
int kg_bce_logits_fwd(const float* score, const float* labels, int n, float* loss_out, float* dscore,
                      void* workspace, size_t workspace_bytes, void* stream);
/* sum of squares of a flat array -> out[0] (deterministic two-stage reduce) */
int kg_sum_squares(const float* x, long long n, float* out, void* workspace, size_t workspace_bytes,
                   void* stream);
int kg_sum(const float* x, long long n, float* out, void* workspace, size_t workspace_bytes,
           void* stream);
/* sum of squares over the first n_valid (device int) rows of x [n_rows, h] -> out[0]; workspace as kg_sum_squares */
int kg_sum_squares_rows(const float* x, int n_rows, int h, const int32_t* n_valid, float* out, void* workspace,
                        size_t workspace_bytes, void* stream);
/* index structures, built once per batch of triplets (integer work, radix sort):
 *   rs_rec  [S]  int4 {a, r, b, t}: the triplets in (r, a) order - runs share w[r] and z[a].  DistMult
 *     is symmetric in its two entities, so {a, b} is {s, o} or, for batches of >= 2^14 triplets, {o, s}
 *     when the object end has the longer run of equal (r, entity) (estimated with a hashed counter
 *     table; negatives that corrupt the subject share (r, o) with their positive)
 *   ent_ptr [n_nodes+1], ent_pack [2S] int4 {other, r, t, 0} in (entity, r) order: for entity v,
 *     every triplet where v is subject (other = object) or object (other = subject)
 * ent_ptr / ent_pack may be NULL: only rs_rec is built (the fused kg_distmult_bce_fwd needs no entity index).
 * Limits: n_nodes < 2^24, n_rels < 2^16. */
size_t kg_triplet_index_workspace_bytes(int n_triplets);
int kg_triplet_index(const int32_t* triplets, int n_triplets, int n_nodes, int n_rels,
                     void* rs_rec, int32_t* ent_ptr, void* ent_pack,
                     void* workspace, size_t workspace_bytes, void* stream);
/* Fused forward of get_loss' prediction term (link_predict.py:74-77) over rs_rec:
 *   score_t = sum_d z[s,d] w[r,d] z[o,d] + shift;  loss_out[0] = mean_t BCE-with-logits(score_t, labels_t)
 *   g_out[t] = dloss/dscore_t = (sigmoid(score_t) - labels_t) / S;  gsum_out[0] = sum_t g_t (d/dshift)
 *   dw[r,:] += sum_{t: r_t = r} g_t z[s_t,:] z[o_t,:]   (dw zero-filled by the caller)
 *   dz[s_t,:] += g_t w[r_t,:] z[o_t,:];  dz[o_t,:] += g_t w[r_t,:] z[s_t,:]   (optional: dz zero-filled by
 *     the caller, or NULL - then kg_distmult_bwd_dz over the entity index gives the same, deterministically)
 *   score_out [S] optional (may be NULL)
 * workspace: kg_distmult_bce_workspace_bytes(S) */
size_t kg_distmult_bce_workspace_bytes(int n_triplets);
int kg_distmult_bce_fwd(const float* z, const float* w, const void* rs_rec, const float* labels,
                        int n_triplets, int h, const float* shift /* device scalar or NULL */,
                        float* score_out, float* g_out, float* dw, float* dz, float* loss_out,
                        float* gsum_out, void* workspace, size_t workspace_bytes, void* stream);
/* dz[v,:] = sum_{(other, r, t) in ent(v)} gscore[t] * w[r,:] * z[other,:]    (no atomics) */
int kg_distmult_bwd_dz(const float* z, const float* w, const float* gscore, const int32_t* ent_ptr,
                       const void* ent_pack, int n_nodes, int h, float* dz, void* stream);

/* Two-pass form of the same backward for a z that does NOT fit L2 (ogbl-wikikg2 shape: 5 GB; new - the reference's
 * index_put(accumulate) backward of kgvae/link_predict.py:57-63 has no counterpart):
 *   kg_triplet_index_trailing   rs_rec as kg_triplet_index, plus the (trailing entity, r)-ordered index of the S
 *                               triplets - trail_ptr [n_nodes + 1], trail_pack [S] int4 {leading entity, r, t, 0};
 *                               "leading" is the end each rs_rec run keeps in registers, "trailing" the other one
 *   kg_distmult_bce_fwd_lead    kg_distmult_bce_fwd with only the leading end's share of dz (accumulated over a run,
 *                               flushed once): no reduction into the random trailing row
 *   kg_distmult_bwd_dz_trailing dz[v] += sum over the triplets whose trailing end is v of g_t w[r_t] z[lead_t]: a
 *                               gather with one owner per row (no atomics, fixed summation order)
 * In DRAM a reduction into a random row is a read-modify-write (4 KB of traffic per 2 KB row), a gather a 2 KB read:
 * 6 KB -> 4 KB of compulsory traffic per scored triplet.  Same workspace sizes as the one-pass entry points;
 * kg_distmult_bce_fwd_lead needs h % 4 == 0, h <= 1024 and 16-byte aligned rows. */
int kg_triplet_index_trailing(const int32_t* triplets, int n_triplets, int n_nodes, int n_rels,
                              void* rs_rec, int32_t* trail_ptr, void* trail_pack,
                              void* workspace, size_t workspace_bytes, void* stream);
int kg_distmult_bce_fwd_lead(const float* z, const float* w, const void* rs_rec, const float* labels,
                             int n_triplets, int h, const float* shift, float* score_out, float* g_out,
                             float* dw, float* dz, float* loss_out, float* gsum_out,
                             void* workspace, size_t workspace_bytes, void* stream);
int kg_distmult_bwd_dz_trailing(const float* z, const float* w, const float* gscore, const int32_t* trail_ptr,
                                const void* trail_pack, int n_nodes, int h, float* dz, void* stream);
/* dw[r,:] += sum_{t: rel_t = r} gscore[t] * z[s_t,:] * z[o_t,:]; dw zero-filled by the caller */
int kg_distmult_bwd_dw(const float* z, const float* gscore, const void* rs_rec, int n_triplets, int h,
                       float* dw, void* stream);

/* ------------------------------------------------------------------------------------
 * a10  all-entity rank evaluation
 * replaces: utils.perturb_and_get_rank kgvae/utils.py:187-221 + sort_and_rank :180-184
 * For each query i: q_i = emb[a_i] * w[r_i]; score_ij = q_i . emb[j] + shift for all j < V;
 * rank_i = #{j : score_ij > score_i,b_i} + #{j < b_i : score_ij == score_i,b_i}  (0-indexed,
 * ties by ascending entity id).  The M x V score matrix is never written to memory: it lives
 * as 128 x 256 tiles in tensor memory (tcgen05.mma on a two-term fp16 split of both operands)
 * and the epilogue counts; pairs the tensor-core value cannot decide are re-scored in fp32.
 * cand_begin/cand_end restrict candidates to an entity shard [begin, end) (multi-GPU: the
 * per-shard counts add up to the rank).
 * filt_ptr/filt_idx (optional, may be NULL): CSR of known-true candidates per query that are
 * removed from the count (filtered setting; the reference itself is raw-only, link_predict.py:7).
 * workspace: kg_distmult_rank_workspace_bytes(n_queries, cand_end - cand_begin, h) bytes.
 * tc_scores: NULL in production; a test hook that receives the tensor-core scores
 *            [n_queries, cand_end - cand_begin] the filter saw.
 * ---------------------------------------------------------------------------------- */
size_t kg_distmult_rank_workspace_bytes(int n_queries, int n_candidates, int h);
int kg_distmult_rank(const float* emb, const float* w, const int32_t* a, const int32_t* r,
                     const int32_t* b, int n_queries, int n_entities, int h,
                     const float* shift /* device scalar or NULL */, int cand_begin, int cand_end,
                     const int32_t* filt_ptr, const int32_t* filt_idx,
                     void* workspace, size_t workspace_bytes, int32_t* ranks, float* tc_scores,
                     void* stream);

/* ------------------------------------------------------------------------------------
 * top-k tail generation
 * replaces: utils.generate kgvae/utils.py:245-288 (the reference scores every entity through the same
 * D x E x V tensor as the evaluation and takes the argmax tail per query; k = 1 there)
 * The k (1..10) highest-scored entities of each query (a_i, r_i) among all n_entities, best first, ties by
 * ascending entity id; scores are the canonical fp32 values of kg_distmult_rank (+ shift).  Same tcgen05
 * score tiles with a top-k epilogue; a finish pass re-scores the listed candidates in fp32 and re-scans any
 * tile the tensor-core rounding could not decide, so the result is exact.
 * ---------------------------------------------------------------------------------- */
size_t kg_distmult_topk_workspace_bytes(int n_queries, int n_entities, int h, int k);
int kg_distmult_topk(const float* emb, const float* w, const int32_t* a, const int32_t* r,
                     int n_queries, int n_entities, int h, const float* shift /* device scalar or NULL */,
                     int k, void* workspace, size_t workspace_bytes, int32_t* out_idx, float* out_score,
                     void* stream);
/* Filtered generation (new; the reference generates from all entities, kgvae/utils.py:245-288): the same, with
 * every entity of query i's list filt_idx[filt_ptr[i] .. filt_ptr[i+1]) (ascending, duplicate-free - the lists of
 * kg_filter_gather) excluded; there is no target to exempt.  Fewer than k unlisted entities: trailing -1 entries.
 * The exclusion happens inside the score-tile epilogue and the finish pass: workspace as kg_distmult_topk. */
int kg_distmult_topk_filtered(const float* emb, const float* w, const int32_t* a, const int32_t* r,
                              int n_queries, int n_entities, int h, const float* shift, int k,
                              const int32_t* filt_ptr, const int32_t* filt_idx, void* workspace,
                              size_t workspace_bytes, int32_t* out_idx, float* out_score, void* stream);
/* Sharded generation (new; multi-GPU): the k best tails among the entities [cand_begin, cand_end) only
 * (0 <= cand_begin <= cand_end <= n_entities), optionally filtered as kg_distmult_topk_filtered (filt_ptr and
 * filt_idx both NULL or both set; the lists hold global ids).  out_idx holds GLOBAL entity ids; the scores are the
 * same canonical bits kg_distmult_topk returns for those entities, so the per-shard lists merge exactly by (score
 * desc, id asc).  Fewer than k eligible entities in the shard (an empty shard included): trailing -1 / -inf.
 * kg_distmult_topk and kg_distmult_topk_filtered are the shard [0, n_entities).
 * workspace: kg_distmult_topk_workspace_bytes(n_queries, cand_end - cand_begin, h, k) bytes. */
int kg_distmult_topk_shard(const float* emb, const float* w, const int32_t* a, const int32_t* r,
                           int n_queries, int n_entities, int h, const float* shift, int k,
                           int cand_begin, int cand_end, const int32_t* filt_ptr /* NULL = unfiltered */,
                           const int32_t* filt_idx, void* workspace, size_t workspace_bytes,
                           int32_t* out_idx, float* out_score, void* stream);

/* ------------------------------------------------------------------------------------
 * filter lists for filtered ranks and filtered generation
 * device counterpart of utils.build_filter, for the filtered forms of perturb_and_get_rank / calc_mrr
 * (kgvae/utils.py:180-221, 293-314) and generate (:245-288) - an extension: the reference is raw-only
 * (kgvae/link_predict.py:7)
 * For a query (a, r): every entity c with (a, r, c) known (KG_FILTER_OBJECT) or (c, r, a) known
 * (KG_FILTER_SUBJECT), ascending and duplicate-free - the filt_ptr / filt_idx CSR of kg_distmult_rank and
 * kg_distmult_topk_filtered.  Entity ids in [0, num_nodes), relation ids in [0, num_rels); a query out of range
 * has an empty list.
 *   kg_filter_table   known triples [T, 3] (s, r, o) -> table [T] (sorted unique keys (a R + r) N + c) and
 *                     table_len (device int).  Needs 2 bits(N) + bits(R) <= 64 (wikikg2: 54).
 *   kg_filter_count   queries (a_i, r_i) -> ptr [M+1]; *total (HOST) = ptr[M], read back once (the call
 *                     synchronises the stream) so that the caller can allocate idx.  Refuses totals >= 2^31.
 *   kg_filter_gather  -> idx [total]
 * ---------------------------------------------------------------------------------- */
#define KG_FILTER_OBJECT 0
#define KG_FILTER_SUBJECT 1
size_t kg_filter_table_workspace_bytes(int n_triples);
int kg_filter_table(const int32_t* triples, int n_triples, int num_nodes, int num_rels, int direction,
                    uint64_t* table, int32_t* table_len, void* workspace, size_t workspace_bytes, void* stream);
size_t kg_filter_count_workspace_bytes(int n_queries);
int kg_filter_count(const uint64_t* table, const int32_t* table_len, int num_nodes, int num_rels,
                    const int32_t* a, const int32_t* r, int n_queries, int32_t* ptr, long long* total,
                    void* workspace, size_t workspace_bytes, void* stream);
int kg_filter_gather(const uint64_t* table, const int32_t* table_len, int num_nodes, int num_rels,
                     const int32_t* a, const int32_t* r, int n_queries, const int32_t* ptr, int32_t* idx,
                     void* stream);

/* Precision of the tensor-core products behind kg_gemm_f32 and kg_distmult_rank (new; the reference runs
 * fp32 library kernels, kgvae/utils.py:200-205, kgvae/flow_network.py:15).  3 (default): the fp32-accurate
 * three-term fp16 split every parity claim is made on.  1: single-product mode - operands rounded to 11
 * significant bits, a third of the MMAs; ranks / outputs then carry that rounding (bench.py reports the mode
 * separately with its measured deviation).  Returns the previous setting. */
int kg_set_tc_terms(int terms);

/* ------------------------------------------------------------------------------------
 * measurement aid (new; no reference counterpart): sustained L2 throughput of this GPU for
 * the access pattern of kg_distmult_bce_fwd - whole fp32 rows of an L2-resident matrix read
 * at random (mode bit 0) and reduced into at random (mode bit 1).  n_ops independent
 * operations; the caller times the call with CUDA events; bytes through L2 =
 * n_ops * 4 * row_floats per enabled direction.  bench.py uses it as the denominator of the
 * "l2" roofline (MEASURED_PEAKS.json only carries HBM and tensor peaks).
 * ---------------------------------------------------------------------------------- */
int kg_probe_l2(const float* src, float* dst, int rows, int row_floats, long long n_ops, int mode,
                float* sink, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* KGVAE_B200_H_ */
