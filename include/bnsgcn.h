/*
 * bnsgcn.h -- C ABI of libbnsgcn.so: the B200 (sm_100a) replacement for the device work the
 * BNS-GCN hot path reaches through DGL / ATen / numpy (SURVEY.md §2.3 K1-K7, §8b).
 *
 * The reference (GATECH-EIC/BNS-GCN, 100 % Python) has no FFI layer of its own: its "operator API"
 * is the set of Python call sites cited beside each entry point below (paths relative to the
 * reference root).  INTEGRATION.md shows the ctypes stub a maintainer would add at each of them.
 *
 * Conventions
 *   - plain C symbols, plain pointers and sizes; no torch / C++ types cross this boundary;
 *   - every pointer marked "device" is a CUDA device pointer owned by the caller (PyTorch owns the
 *     tensors; the library never frees or reallocates caller memory);
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing synchronises
 *     the host except bns_graph_create / bns_graph_transpose (setup) and where stated;
 *   - return value: 0 = ok, negative = error (BNS_E_*); bns_last_error() gives the message of the
 *     calling thread's most recent failure;
 *   - after *_create the library allocates nothing: scratch space is passed in (`ws`, sized by the
 *     matching *_workspace_bytes query);
 *   - thread-compatible: distinct handles may be used from distinct threads concurrently.
 *   - feature matrices are row-major f32; graph ids int32 on device (train.py:71-73 uses int32
 *     graphs), row offsets int64, exchanged index lists int64 (train.py:233-234, utils.py:171).
 */
#ifndef BNSGCN_H_
#define BNSGCN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BNS_OK            0
#define BNS_E_INVALID    (-1)   /* bad argument (null pointer, negative size, misaligned leading dim) */
#define BNS_E_CUDA       (-2)   /* a CUDA runtime call failed; message holds cudaGetErrorString */
#define BNS_E_WORKSPACE  (-3)   /* workspace too small */
#define BNS_E_UNSUPPORTED (-4)

#define BNS_ABI_VERSION 3

typedef struct bns_graph bns_graph_t;   /* opaque: a static CSR matrix resident in HBM */
typedef struct bns_p2p   bns_p2p_t;     /* opaque: peer-mapped exchange slabs of one rank */
typedef struct bns_ctx   bns_ctx_t;     /* opaque: one rank's communicator (NCCL) */

int         bns_abi_version(void);
const char *bns_last_error(void);
/* Number of kernels of this library enqueued so far by this process (bench.py reports the delta as gpu_launches). */
uint64_t    bns_launch_count(void);
/* Name, SM count, L2 bytes of the current device (for bench.py's grid / roofline bookkeeping). */
int         bns_device_info(char *name, size_t name_len, int *sm_count, int64_t *l2_bytes, int *cc_major, int *cc_minor);

/* ------------------------------------------------------------------------------------------------
 * Static graphs.  Replaces the per-epoch dgl.heterograph rebuild of train.py:256-281
 * (construct_graph) and DGL's lazy COO->CSR/CSC conversion: a graph is built ONCE, per-epoch
 * sampling only changes the small `col_map` / `row_map` arrays given to bns_spmm_sum_f32.
 *
 * bns_graph_create copies a device CSR (row r's entries are indices[indptr[r] .. indptr[r+1])) and
 * precomputes the nnz-balanced work decomposition (rows are cut into chunks of <= chunk_nnz
 * entries; rows longer than a chunk are combined by a deterministic second pass).
 *   n_rows, n_cols : matrix shape; every index must lie in [0, n_cols)
 *   chunk_nnz      : 0 = library default
 * ----------------------------------------------------------------------------------------------*/
int bns_graph_create(bns_graph_t **out, int64_t n_rows, int64_t n_cols, int64_t nnz,
                     const int64_t *indptr /*device [n_rows+1]*/, const int32_t *indices /*device [nnz]*/,
                     int32_t chunk_nnz, void *stream);
/* CSR of the reversed graph (what autograd needs for K1b, SURVEY §2.3): out[c] lists the rows r with
 * (r, c) in g, ascending.  Built once, on the device (radix sort). */
int bns_graph_transpose(const bns_graph_t *g, bns_graph_t **out, void *stream);
int bns_graph_destroy(bns_graph_t *g);
int bns_graph_info(const bns_graph_t *g, int64_t *n_rows, int64_t *n_cols, int64_t *nnz,
                   int64_t *n_chunks, int64_t *n_split_rows);
/* For a graph made by bns_graph_transpose: perm_out[k] (device [nnz]) = index, in the SOURCE graph's CSR order, of
 * the entry that became entry k of the transpose -- carries per-entry weights across (w_T[k] = w[perm[k]]). */
int bns_graph_copy_perm(const bns_graph_t *gT, int32_t *perm_out, void *stream);
/* Copy the library-owned CSR into caller buffers (device [n_rows+1] / [nnz]); for tests and tools. */
int bns_graph_copy_csr(const bns_graph_t *g, int64_t *indptr_out, int32_t *indices_out, void *stream);

/* ------------------------------------------------------------------------------------------------
 * K1 / K1b / K2: the aggregation.  Replaces
 *     graph['_E'].update_all(fn.copy_u('h','m'), fn.sum('m','h'))        module/layer.py:35-37, 88-90
 *     ... / degs, feat / out_norm, ... / in_norm                         module/layer.py:34, 38, 91
 * and their autograd transposes, with
 *     Y[orow(r), :] = (accumulate ? Y[orow(r), :] : 0)
 *                     + row_scale[r] * sum_{k in row r, xrow(c_k) >= 0} col_scale[c_k] * X[xrow(c_k), :]
 *   xrow(c) = c                       if c <  n_direct
 *           = col_map[c - n_direct]   otherwise (-1 = entry skipped: an unsampled halo node)
 *   orow(r) = r  if row_map == NULL, else row_map[r]  (-1 = row skipped)
 * row_scale / col_scale / row_map / col_map may be NULL (= 1 / identity; col_map == NULL means
 * n_direct = n_cols).  All f32; summation order inside a row is the CSR order (deterministic).
 *   X  [*, F] with leading dimension ldx (floats); Y [*, F] with ldy.
 * The 16-byte vector path needs F % 4 == 0, ldx % 4 == 0, ldy % 4 == 0 and 16-byte aligned X, Y;
 * anything else takes the scalar path (same results).
 * ws: scratch of at least bns_spmm_workspace_bytes(g, F) bytes (0 when no row is split).
 * L2 blocking: the feature dimension is processed in column slabs (256/128/64/32 floats) picked so that
 * x_rows * slab * 4 bytes stays resident in L2 (override: slab_hint, or env BNS_SPMM_SLAB).
 * ----------------------------------------------------------------------------------------------*/
size_t bns_spmm_workspace_bytes(const bns_graph_t *g, int64_t F);
int bns_spmm_sum_f32(const bns_graph_t *g,
                     const float *X, int64_t ldx, int64_t F,
                     float *Y, int64_t ldy,
                     const float *row_scale /*device [n_rows] or NULL*/,
                     const float *col_scale /*device [n_cols] or NULL*/,
                     const float *edge_weight /*device [nnz], CSR order, or NULL: multiplies entry k's source row
                                                (GAT attention, u_mul_e + sum of dgl.nn.GATConv)*/,
                     const int32_t *row_map /*device [n_rows] or NULL*/,
                     const int32_t *col_map /*device [n_cols - n_direct] or NULL*/, int64_t n_direct,
                     int64_t x_rows /*rows of X that can be referenced (0 = n_cols); sizes the L2 blocking*/,
                     int32_t slab_hint /*0 = automatic; 256 | 128 | 64 | 32 forces the column-slab width*/,
                     int accumulate, void *ws, size_t ws_bytes, void *stream);

/* ------------------------------------------------------------------------------------------------
 * K8: the dense layers themselves.  Replaces, for 2-D f32 operands,
 *     self.linear(feat) / self.linear1(feat) + self.linear2(ah)      module/layer.py:30, 38, 83, 92  (forward)
 * and what autograd runs for them (grad_input = dY W, grad_weight = dY^T X) with hand-written tcgen05 kernels:
 * kind::tf32 MMAs accumulating in TMEM, operands staged by TMA (SWIZZLE_128B), and the 3xTF32 operand split
 * (hi = tf32(x), lo = x - hi; hi*hi + hi*lo + lo*hi) done in shared memory inside the pipeline, so the result is
 * f32-accurate (~2^-21 relative per product) while every operand byte crosses HBM/L2 once (csrc/dense_tc.cuh).
 *
 * bns_dense_tn_3xtf32:  C[M, N] = A[M, K] * B[N, K]^T (+ bias[N]) (+ addend[M, N]);  A, B, C row-major with leading
 *   dimensions lda, ldb, ldc (floats).  Forward: A = X, B = weight; `addend` fuses the "+" of
 *   linear1(feat) + linear2(ah) (module/layer.py:92) into the epilogue.  Input gradient: A = dY, B = weight^T (a
 *   contiguous copy).
 * bns_dense_nt_3xtf32:  C[N1, N2] = A[R, N1]^T * B[R, N2]  (contraction over the R rows, split across CTAs and
 *   combined in split order -- deterministic).  Weight gradient: A = dY, B = X.  ws: at least
 *   bns_dense_nt_workspace_bytes(R, N1, N2) bytes.
 * All pointers 16-byte aligned, leading dimensions multiples of 4 (and N2 % 4 == 0); anything else returns
 * BNS_E_INVALID and the caller uses the library GEMM.
 * ----------------------------------------------------------------------------------------------*/
int    bns_dense_tn_3xtf32(const float *A, int64_t lda, const float *B, int64_t ldb, const float *bias /*device [N] or NULL*/,
                           const float *addend /*device [M, N] with leading dimension ldadd, or NULL; may alias C*/, int64_t ldadd,
                           const float *row_scale /*device [M] or NULL: C[r, :] = (A B^T + bias + addend)[r, :] * row_scale[r]
                                                    (the 1/deg pre-scale of the aggregation's backward, module/layer.py:91)*/,
                           float *C, int64_t ldc, int64_t M, int64_t N, int64_t K, void *stream);
size_t bns_dense_nt_workspace_bytes(int64_t R, int64_t N1, int64_t N2);
int    bns_dense_nt_3xtf32(const float *A, int64_t lda, const float *B, int64_t ldb, float *C, int64_t ldc,
                           int64_t R, int64_t N1, int64_t N2, void *ws, size_t ws_bytes, void *stream);
/* Bias gradient of the same layers (autograd's dY.sum(0)): out[c] = sum_r X[r, c], two deterministic passes.
 * cols % 4 == 0, cols <= 1024, ld % 4 == 0, 16-byte aligned; ws >= bns_colsum_workspace_bytes(cols). */
size_t bns_colsum_workspace_bytes(int64_t cols);
int    bns_colsum_f32(const float *X, int64_t ld, int64_t rows, int64_t cols, float *out,
                      float *out2 /*optional second destination (linear1.bias and linear2.bias share dY.sum(0))*/, void *ws,
                      size_t ws_bytes, void *stream);

/* ------------------------------------------------------------------------------------------------
 * K10 (GAT, module/model.py:96-132 via dgl.nn.GATConv): the attention gradient.  For every entry k of row r:
 *     out[k * ldo] = < A[arow(r), :F], B[xrow(c_k), :F] >      (0 when the row or the entry is skipped)
 * arow / xrow as in bns_spmm_sum_f32 (row_map / col_map / n_direct).  F % 4 == 0, F <= 1024, 16-byte aligned rows.
 * With bns_spmm_sum_f32(edge_weight) and the transpose permutation this is all GATConv needs besides elementwise
 * work on per-entry vectors: forward  rst = A_w ft,  backward  d ft = A_w^T d rst,  d w = sddmm(d rst, ft).
 * ----------------------------------------------------------------------------------------------*/
int bns_sddmm_dot_f32(const bns_graph_t *g, const float *A, int64_t lda, const float *B, int64_t ldb, int64_t F,
                      const int32_t *row_map, const int32_t *col_map, int64_t n_direct, float *out, int64_t ldo,
                      void *stream);

/* ------------------------------------------------------------------------------------------------
 * K3 / K4 / K5: boundary pack / concat / scatter.  helper/feature_buffer.py:
 *   :117  send_cpu[right].copy_(send_gpu[self._selected[right]] / self._ratio[right])
 *   :85-91 __feat_concat  (cat([feat, recv_0, ...]))
 *   :129  send_gpu[self._selected[idx]] += recv / self._ratio[idx]
 * out[i, :] = H[idx[i], :] / div        (true division, as the reference)
 * G[idx[i], :] += src[i, :] / div       (idx must not repeat inside one call; calls on one stream
 *                                         are ordered, which is how the reference orders peers)
 * ----------------------------------------------------------------------------------------------*/
int bns_gather_div_f32(const float *H, int64_t ldh, int64_t F, const int64_t *idx /*device [k]*/, int64_t k,
                       float div, float *out, int64_t ldo, void *stream);
int bns_scatter_add_div_f32(float *G, int64_t ldg, int64_t F, const int64_t *idx /*device [k]*/, int64_t k,
                            float div, const float *src, int64_t lds, void *stream);
/* dst[r, :F] = src[r, :F] for r < n_rows (the "inner" block of the concat buffer). */
int bns_copy_rows_f32(const float *src, int64_t lds, float *dst, int64_t ldd, int64_t n_rows, int64_t F, void *stream);

/* ------------------------------------------------------------------------------------------------
 * K6: boundary-node sampling.  Replaces train.py:225-236 (select_node):
 *     idx = np.random.choice(b.shape[0], send_size[i], replace=False);  selected = boundary[i][idx]
 * i.e. a uniformly random ORDERED k-subset per peer.  All peers are drawn by one call:
 *   boundary_cat : the sorted boundary lists of the n_seg peers, concatenated (device, int64 [B])
 *   seg_begin    : device int64 [n_seg+1], boundary list s is boundary_cat[seg_begin[s] .. seg_begin[s+1])
 *   out_begin    : device int64 [n_seg+1], prefix sums of the sample sizes k_s (k_s <= b_s)
 *   selected     : device int64 [K_total], peer s's sample is selected[out_begin[s] .. out_begin[s+1])
 * Element i of boundary_cat gets the key  (s << 56) | r56(i),  r56 = the top 56 bits of
 * Philox4x32-10(counter = (i_lo, i_hi, offset_lo, offset_hi), key = (seed_lo, seed_hi)) words 0,1;
 * a stable radix sort orders each segment by key and the first k_s entries are the sample.
 * Counter-based => reproducible: the oracle replays it bit for bit (oracle/philox.py).
 * ----------------------------------------------------------------------------------------------*/
size_t bns_sample_workspace_bytes(int64_t B);
int bns_sample_boundary(const int64_t *boundary_cat, const int64_t *seg_begin, const int64_t *out_begin,
                        int32_t n_seg, int64_t B, int64_t K_total, uint64_t seed, uint64_t offset,
                        const uint64_t *offset_dev /*device, optional: added to `offset` at run time, so that a
                                                     captured CUDA graph draws a new sample on every replay*/,
                        int64_t *selected, void *ws, size_t ws_bytes, void *stream);

/* ------------------------------------------------------------------------------------------------
 * K7: per-epoch graph "rebuild".  Replaces train.py:256-281 (construct_graph) and 245-253
 * (construct_out_norm): instead of building a new heterograph, record where each sampled halo node's
 * row lives in the receive slab:
 *     slot[pos[one_hops[k]] - n_in] = slab_offset + k        k = 0 .. r-1
 * (`pos` = get_pos() of train.py:90-104: owner-local id -> my local node id, -1 if not my halo).
 * Call bns_fill_i32(slot, n_halo, -1) first, then once per peer.
 * ----------------------------------------------------------------------------------------------*/
int bns_fill_i32(int32_t *dst, int64_t n, int32_t value, void *stream);
int bns_halo_slot_update(const int64_t *pos /*device [part size of the peer]*/, const int64_t *one_hops /*device [r]*/,
                         int64_t r, int64_t n_in, int32_t slab_offset, int32_t *slot /*device [n_halo]*/, void *stream);

/* ------------------------------------------------------------------------------------------------
 * K9 (fused): LayerNorm -> ReLU -> dropout between two layers.  Replaces the three ATen ops of
 * module/model.py:88-91 (`h = self.norm[i](h); h = self.activation(h)`) and :45/:80 of the next iteration
 * (`h = self.dropout(h)`), forward and backward, in one pass each:
 *     y = dropout_p( relu( (x - mean) * rstd * gamma + beta ) )        mean / biased var over the F columns
 * The dropout mask is Philox4x32-10(counter = (row, vector, offset), key = seed) -- regenerated, not stored, in
 * backward; offset_dev (optional, device) is added to offset at run time (CUDA-graph replays).  F % 4 == 0,
 * F <= 1024.  Backward also returns dgamma / dbeta (column sums, fixed summation order: deterministic);
 * ws: bns_ln_bwd_workspace_bytes(F) bytes.
 * ----------------------------------------------------------------------------------------------*/
size_t bns_ln_bwd_workspace_bytes(int64_t F);
int bns_ln_relu_dropout_fwd_f32(const float *x, int64_t ldx, int64_t n, int64_t F, const float *gamma,
                                const float *beta, float eps, float p, uint64_t seed, uint64_t offset,
                                const uint64_t *offset_dev, float *y, int64_t ldy, float *mean /*[n]*/,
                                float *rstd /*[n]*/, void *stream);
int bns_ln_relu_dropout_bwd_f32(const float *dy, int64_t lddy, const float *x, int64_t ldx, int64_t n, int64_t F,
                                const float *gamma, const float *beta, const float *mean, const float *rstd,
                                float eps, float p, uint64_t seed, uint64_t offset, const uint64_t *offset_dev,
                                float *dx, int64_t lddx, float *dgamma /*[F]*/, float *dbeta /*[F]*/, void *ws,
                                size_t ws_bytes, void *stream);

/* ------------------------------------------------------------------------------------------------
 * C1/C2 fused with K3/K5: the boundary exchange over peer-mapped memory (NVLink 5 / NVSwitch).
 * Replaces Buffer.__gloo_all_to_all / __mpi_all_to_all (helper/feature_buffer.py:101-153): the pack
 * kernel of rank a stores  H[selected_b] / ratio_b  straight into rank b's receive slab, then raises a
 * flag in b's memory; b's stream waits on the flag.  No staging buffer, no host round trip.
 * One bns_p2p_t per rank; slabs are cudaMalloc'd by the library so that they can be exported with
 * cudaIpcGetMemHandle (processes) or shared by pointer (ranks that are threads of one process).
 * ----------------------------------------------------------------------------------------------*/
#define BNS_P2P_HANDLE_BYTES 64
int bns_p2p_create(bns_p2p_t **out, int32_t rank, int32_t world, size_t slab_bytes, int32_t n_flags);
int bns_p2p_destroy(bns_p2p_t *p);
/* base of this rank's slab / flag block (device pointers, valid in this process) */
int bns_p2p_local(const bns_p2p_t *p, void **slab, void **flags, size_t *slab_bytes);
/* IPC export / import (multi-process).  handle_out: BNS_P2P_HANDLE_BYTES bytes for the slab followed by
 * BNS_P2P_HANDLE_BYTES bytes for the flags. */
int bns_p2p_export(const bns_p2p_t *p, void *handle_out /*2*BNS_P2P_HANDLE_BYTES*/);
int bns_p2p_import(bns_p2p_t *p, int32_t peer, const void *handle /*2*BNS_P2P_HANDLE_BYTES*/, size_t peer_slab_bytes);
/* In-process peers (threads): register the peer's pointers directly. */
int bns_p2p_set_peer(bns_p2p_t *p, int32_t peer, void *slab, void *flags, size_t peer_slab_bytes);
/* remote_rows[i, :F] (in peer's slab at byte offset remote_off, leading dim ld_remote floats)
 *     = H[idx[i], :F] / div   for i < k   (idx == NULL: rows i of H, used for the gradient return trip);
 * then, after a system-scope fence, peer.flags[flag_index] = flag_value (release). */
int bns_p2p_put_rows_f32(bns_p2p_t *p, int32_t peer, size_t remote_off, int64_t ld_remote,
                         const float *H, int64_t ldh, int64_t F, const int64_t *idx, int64_t k, float div,
                         int32_t flag_index, uint64_t flag_value,
                         const uint64_t *flag_value_dev /*device, optional: added to flag_value at run time (graph replays)*/,
                         void *stream);
/* Enqueue a wait on `stream` until this rank's flags[flag_index] >= flag_value (acquire).  The spin is bounded
 * (20 s): a peer that never signals traps the kernel (a loud CUDA error) instead of hanging the device. */
int bns_p2p_wait_flag(bns_p2p_t *p, int32_t flag_index, uint64_t flag_value, const uint64_t *flag_value_dev,
                      void *stream);


/* ================================================================================================
 * ABI 2: the rest of the epoch (train.py:385-425) as ONE launch per step instead of one per peer / per parameter /
 * per ATen op.  At 8 partitions the round-1 epoch spent ~59 % of its time in such launches.
 * ================================================================================================*/
#define BNS_MAX_PEERS 16

/* ------------------------------------------------------------------------------------------------
 * K7': slot map of ALL peers + the inverse maps the gradient scatter walks, one memset + one kernel.  Replaces the
 * per-peer loop of train.py:256-281 (construct_graph) done by bns_fill_i32 + bns_halo_slot_update x (P-1):
 *     slot[pos_s[one_hops_cat[k]] - n_in] = k                         k over the concatenated received id lists
 *     inv_s[selected_cat[i]] = i - sel_begin[s]                       i over the concatenated sampled id lists
 * Segments = the peers in ascending order, self skipped.  [fill_base, +fill_bytes) -- the allocation that holds `slot`
 * and every inv_s -- is set to -1 first.
 * ----------------------------------------------------------------------------------------------*/
typedef struct bns_epoch_maps {
    int32_t n_seg;
    int64_t sel_begin[BNS_MAX_PEERS + 1];
    int64_t hop_begin[BNS_MAX_PEERS + 1];
    const int64_t *pos[BNS_MAX_PEERS];      /* device: get_pos() of train.py:90-104 */
    int32_t *inv[BNS_MAX_PEERS];            /* device [n_in] each, may be NULL */
    const int64_t *selected_cat, *one_hops_cat;
    int32_t *slot;                          /* device [n_halo] */
    int64_t n_in;
} bns_epoch_maps;
int bns_epoch_maps_update(const bns_epoch_maps *maps /*host*/, void *fill_base, size_t fill_bytes, void *stream);

/* ------------------------------------------------------------------------------------------------
 * K1 on the SAMPLED halo only.  bns_graph_compact_cols rewrites, once per epoch, the column ids of a column-mapped
 * matrix (A_out with col_map = slot): chunk by chunk, the entries whose column is sampled are moved -- already mapped to
 * rows of X, CSR order kept -- to the front of the chunk's own index range in `cidx`, their number goes to
 * `chunk_cnt`; bns_spmm_compact_f32 then runs the plain kernel over exactly those entries.  Same numbers added in the
 * same order as bns_spmm_sum_f32(col_map): bit-identical results, work proportional to the sample
 * (train.py:256-281 builds the sampled graph per epoch for the same reason).
 * ----------------------------------------------------------------------------------------------*/
int bns_graph_compact_cols(const bns_graph_t *g, const int32_t *col_map, int64_t n_direct,
                           const float *col_scale /*device [n_cols] or NULL: gathered per live entry into cw*/,
                           int32_t *cidx /*device [nnz]*/, float *cw /*device [nnz] or NULL*/,
                           int32_t *cpos /*device [nnz] or NULL: position of each live entry in the CSR (GAT keeps its
                                           per-entry attention at those positions)*/,
                           int32_t *chunk_cnt /*device [n_chunks]*/, void *stream);
int bns_spmm_compact_f32(const bns_graph_t *g, const int32_t *cidx, const float *cw /*per compacted entry, or NULL*/,
                         int64_t cw_ld /*stride of cw in floats (1; heads for GAT's [nnz, heads] attention)*/,
                         const int32_t *chunk_cnt, const float *X, int64_t ldx, int64_t F, float *Y, int64_t ldy,
                         const float *row_scale, int64_t x_rows, int32_t slab_hint, int accumulate, void *ws, size_t ws_bytes,
                         void *stream);

/* ------------------------------------------------------------------------------------------------
 * K10 staged: the attention of dgl.nn.GATConv (module/model.py:96-132; DGL 0.9 python/dgl/nn/pytorch/conv/gatconv.py):
 *     e_uv = leaky_relu(el_u + er_v);  p = edge_softmax(e) over each destination's in-entries;  a = attn_drop(p);
 *     rst_v = sum_u a_uv ft_u                     for all `heads` at once.
 * The entries of row v are those of a_in followed by the SAMPLED ones of a_out (cidx / chunk_cnt / cpos from
 * bns_graph_compact_cols with col_map = slot, n_direct = 0; halo source k reads ft row x_halo_base + k).
 *   el [n_u, heads], er [n_in, heads], heads <= 8.  P_in [nnz(a_in), heads] / P_out [nnz(a_out), heads]: the
 *   probabilities, stored at the ORIGINAL entry positions, kept for the backward.  Dropout: Philox4x32-10(counter =
 *   (entry, head), key = seed, offset [+ *offset_dev]), regenerated in backward.
 * Each stage keeps thousands of independent gathers in flight:
 *   forward   bns_gat_scores_f32 -- scalars only, one warp per destination row: P and the dropped attention
 *             W = p * mask / (1 - q) at the original positions, W_out_compact at the compacted positions -- then
 *             rst = W ft by bns_spmm_weighted_f32 / bns_spmm_compact_f32, one head per call;
 *   backward  bns_sddmm_dot_f32 writes d a' = <d rst_v, ft_u> into dE_in / dE_out (same layout as P);
 *             bns_gat_softmax_bwd_f32 turns it into d e in place and writes d er [n_in, heads];
 *             bns_gat_colsum_f32 (on a_in_t, then on a_out_t with row_map = slot): d el_u = sum over column u of d e;
 *             bns_spmm_weighted_f32: d ft = W^T d rst, one head per call, the attention read through the transpose's
 *             permutation.
 * ----------------------------------------------------------------------------------------------*/
int bns_gat_scores_f32(const bns_graph_t *a_in, const bns_graph_t *a_out, const int32_t *cidx, const int32_t *chunk_cnt,
                       const int32_t *cpos, int64_t x_halo_base, int32_t heads, const float *el, const float *er,
                       float negative_slope, float p_drop, uint64_t seed, uint64_t offset, const uint64_t *offset_dev,
                       float *P_in, float *P_out, float *W_in /*NULL when p_drop == 0*/, float *W_out, float *W_out_compact,
                       void *stream);
int bns_gat_softmax_bwd_f32(const bns_graph_t *a_in, const bns_graph_t *a_out, const int32_t *cidx, const int32_t *chunk_cnt,
                            const int32_t *cpos, int64_t x_halo_base, int32_t heads, const float *el, const float *er,
                            float negative_slope, float p_drop, uint64_t seed, uint64_t offset, const uint64_t *offset_dev,
                            const float *P_in, const float *P_out, float *dE_in, float *dE_out, float *d_er, void *stream);
/* el / er of GATConv (module/model.py:102; DGL 0.9 gatconv.py: el = (feat_src * attn_l).sum(-1), er likewise): out[r, h] = <X[r, h*Fo:(h+1)*Fo], attn[h, :]>, and its backward: dX[r, h, :] (+)= s[r, h] * attn[h, :],
 * d_attn[h, :] = sum_r s[r, h] * X[r, h, :] (deterministic).  ws: bns_colsum_workspace_bytes(heads * Fo). */
int bns_gat_proj_f32(const float *X, int64_t ldx, int64_t rows, int32_t heads, int32_t Fo, const float *attn, float *out,
                     void *stream);
int bns_gat_proj_bwd_f32(const float *X, int64_t ldx, int64_t rows, int32_t heads, int32_t Fo, const float *attn,
                         const float *s, float *dX, int64_t lddx, int accumulate, float *d_attn, void *ws, size_t ws_bytes,
                         void *stream);
int bns_gat_colsum_f32(const bns_graph_t *gT, const float *dE, int32_t heads, const int32_t *row_map, int64_t out_base,
                       float *d_el, void *stream);
int bns_spmm_weighted_f32(const bns_graph_t *g, const float *X, int64_t ldx, int64_t F, float *Y, int64_t ldy,
                          const float *weights, int64_t ldw, int perm_from_transpose, const int32_t *row_map, int64_t x_rows,
                          int accumulate, void *ws, size_t ws_bytes, void *stream);

/* ------------------------------------------------------------------------------------------------
 * C1/C2 + K3/K5 for ALL peers at once (helper/feature_buffer.py:101-129).
 * bns_p2p_put_all_f32: segment s sends rows [row_begin[s], row_begin[s+1]) of the concatenated send list to peer[s]:
 *     remote_s[i, :F] = H[idx_cat[row_begin[s] + i], :F] / div[s]      (idx_cat == NULL: H[src_begin[s] + i, :F])
 * into the peer's slab at byte offset remote_off[s]; after the last row of the LAUNCH every peer's flags[flag_index]
 * is set to flag_value (+ *flag_value_dev) with a system-scope release.  ticket_index < world + 16 picks the completion
 * counter; launches that share one must be stream-ordered.
 * bns_p2p_put_ids_i64: the same for the sampled id lists (data_transfer(..., tag=NODE), helper/utils.py:187-213).
 * bns_p2p_wait_all: one kernel that waits for n flags of this rank (bounded spin, 20 s -> trap).
 * bns_scatter_rows_all_f32: G[r, :] += recv_s[inv_s[r], :] / div[s] for every segment s IN ORDER and every row r with
 *     inv_s[r] >= 0 -- the P-1 scatter-adds of :129 in the reference's peer order, race-free in one launch.
 * ----------------------------------------------------------------------------------------------*/
typedef struct bns_put_all {
    int32_t n_seg;
    int64_t row_begin[BNS_MAX_PEERS + 1];
    int32_t peer[BNS_MAX_PEERS];
    uint64_t remote_off[BNS_MAX_PEERS];
    int64_t src_begin[BNS_MAX_PEERS];
    float div[BNS_MAX_PEERS];
} bns_put_all;
int bns_p2p_put_all_f32(bns_p2p_t *p, const bns_put_all *segs /*host*/, int64_t ld_remote, const float *H, int64_t ldh,
                        int64_t F, const int64_t *idx_cat, int32_t flag_index, int32_t ticket_index, uint64_t flag_value,
                        const uint64_t *flag_value_dev, void *stream);
int bns_p2p_put_ids_i64(bns_p2p_t *p, int32_t n_seg, const int64_t *begin /*host [n_seg+1]*/, const int32_t *peers /*host*/,
                        const uint64_t *remote_off /*host*/, const int64_t *ids_cat /*device*/, int32_t flag_index,
                        int32_t ticket_index, uint64_t flag_value, const uint64_t *flag_value_dev, void *stream);
int bns_p2p_wait_all(bns_p2p_t *p, int32_t n, const int32_t *flag_indices /*host*/, uint64_t flag_value,
                     const uint64_t *flag_value_dev, void *stream);
int bns_scatter_rows_all_f32(float *G, int64_t ldg, int64_t n_rows, int64_t F, int32_t n_seg,
                             const int32_t *const *inv /*host array of device pointers*/,
                             const float *const *recv /*host array of device pointers*/, int64_t ld_recv,
                             const float *div /*host*/, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Loss and its gradient in one launch.  Replaces train.py:406-408 for the two losses of train.py:358-361:
 *     loss = CrossEntropyLoss(reduction='sum')(logits[train_mask], labels[train_mask])          (labels != NULL)
 *     loss = BCEWithLogitsLoss(reduction='sum')(logits[train_mask], labels[train_mask])        (labels_f != NULL)
 * dlogits[r, :n_class] = d loss / d logits[r, :] * grad_scale for train rows, 0 for the others and for the pad columns
 * [n_class, n_cols_out).  grad_scale = 1 / n_train folds helper/reducer.py:34 (grad /= n_train) into the source of
 * every gradient.  The loss is summed block by block in a fixed order (deterministic).  ws: bns_xent_workspace_bytes()
 * bytes, zeroed ONCE by the caller.
 * ----------------------------------------------------------------------------------------------*/
size_t bns_xent_workspace_bytes(void);
int bns_xent_f32(const float *logits, int64_t ld, int64_t n_rows, int32_t n_class, const int64_t *labels,
                 const float *labels_f, int64_t ldl, const uint8_t *mask /*device bool [n_rows] or NULL*/, float grad_scale,
                 float *loss_out /*device [1]*/, float *dlogits, int64_t ldd, int32_t n_cols_out, void *ws, size_t ws_bytes,
                 void *stream);

/* ------------------------------------------------------------------------------------------------
 * torch.optim.Adam (train.py:362, :413) over ONE flat parameter arena: every parameter, its gradient and both moments
 * live at the same offsets of four flat buffers, so the step is one launch (torch: ~15 multi-tensor launches).
 *     g += weight_decay * p;  m += (1 - b1) (g - m);  v = b2 v + (1 - b2) g^2;
 *     p -= lr / (1 - b1^t) * m / (sqrt(v) / sqrt(1 - b2^t) + eps),        t = *step_dev + 1
 * bns_derive_refresh (enqueue right after): refreshes the table of derived parameters -- cached W^T for the input
 * gradients, bias sums -- and advances *step_dev.  Entry layout: bns_derive_entry, table in device memory.
 * ----------------------------------------------------------------------------------------------*/
typedef struct bns_derive_entry {
    int32_t op;        /* 0: dst[c * ld_dst + r] = a[r * ld_a + c], r < rows, c < cols;  1: dst[i] = a[i] + b[i], i < rows */
    int32_t rows, cols, ld_a, ld_dst, pad_;
    const float *a, *b;
    float *dst;
} bns_derive_entry;
size_t bns_derive_entry_bytes(void);
int bns_adam_step_f32(float *param, const float *grad, float *exp_avg, float *exp_avg_sq, int64_t n, float lr, float beta1,
                      float beta2, float eps, float weight_decay, const int64_t *step_dev, void *stream);
int bns_derive_refresh(const void *table_dev, int32_t n_entries, int64_t *step_dev, void *stream);

/* ------------------------------------------------------------------------------------------------
 * SyncBatchNorm (--norm batch; module/sync_bn.py:7-56): batch statistics over every partition.
 * Forward:  bns_bn_colsums_f32(mode 0) -> [sum x | sum x^2] per column; the caller all-reduces the packed [2F] vector;
 *           bns_bn_apply_f32: mean = S1 / n, var = (S2 - mean S1) / n (n = whole_size, the global TRAIN count:
 *           sync_bn.py:19-20 with model.py:39), y = (x - mean) / sqrt(var + eps) * weight + bias, running statistics
 *           moved by `momentum`, mean / rstd kept for the backward.
 * Backward: bns_bn_colsums_f32(mode 1) -> [sum dy | sum dy x_hat]; packed all-reduce; these ARE d bias / d weight;
 *           bns_bn_bwd_f32: dx = (weight / n) / std * (n dy - d bias - x_hat d weight)        (sync_bn.py:51-54).
 * Two collectives per layer and step instead of four, three passes over the activations instead of ~12.
 * F % 4 == 0, F <= 1024, 16-byte aligned rows.
 * ----------------------------------------------------------------------------------------------*/
size_t bns_bn_workspace_bytes(int64_t F);
int bns_bn_colsums_f32(int mode, const float *A, int64_t lda, const float *X, int64_t ldx, int64_t rows, int64_t F,
                       const float *mean, const float *rstd, float *out /*device [2F]*/, void *ws, size_t ws_bytes, void *stream);
int bns_bn_apply_f32(const float *x, int64_t ldx, int64_t rows, int64_t F, const float *sums /*device [2F]*/, float whole_size,
                     float eps, const float *weight, const float *bias, float momentum, float *running_mean /*or NULL*/,
                     float *running_var, float *y, int64_t ldy, float *mean_out /*[F]*/, float *rstd_out /*[F]*/, void *stream);
int bns_bn_bwd_f32(const float *dy, int64_t lddy, const float *x, int64_t ldx, int64_t rows, int64_t F, const float *mean,
                   const float *rstd, const float *weight, const float *sums /*device [2F]*/, float whole_size, float *dx,
                   int64_t lddx, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Collectives (SURVEY 8b).  One context per rank / GPU; NCCL underneath, resolved at run time (dlopen).
 * Bootstrap: rank 0 calls bns_comm_unique_id and hands the BNS_COMM_ID_BYTES bytes to the other ranks by any
 * out-of-band means (the reference rendezvouses over TCP, train.py:459-468); every rank then calls bns_ctx_create.
 *   bns_allreduce_sum_f32   helper/reducer.py:28-49: the weight gradients, as ONE flat bucket, in place
 *   bns_alltoallv_i64       helper/utils.py:187-213 data_transfer(..., tag=NODE): the sampled id lists
 *   bns_alltoallv_f32       helper/feature_buffer.py:101-153: boundary rows, staged transport (the peer-mapped transport
 *                           -- bns_p2p_* -- needs no collective at all)
 * counts / offsets: host arrays [world], in rows of `width` elements; the entry of the own rank is ignored.
 * ----------------------------------------------------------------------------------------------*/
#define BNS_COMM_ID_BYTES 128
int bns_comm_unique_id(void *id_out /*host, BNS_COMM_ID_BYTES*/);
int bns_ctx_create(bns_ctx_t **out, int32_t rank, int32_t world, const void *unique_id /*host, BNS_COMM_ID_BYTES*/);
int bns_ctx_destroy(bns_ctx_t *c);
int bns_allreduce_sum_f32(bns_ctx_t *c, float *buf /*device*/, int64_t n, void *stream);
int bns_alltoallv_f32(bns_ctx_t *c, const float *send, const int64_t *send_counts, const int64_t *send_offsets, float *recv,
                      const int64_t *recv_counts, const int64_t *recv_offsets, int64_t width, void *stream);
int bns_alltoallv_i64(bns_ctx_t *c, const int64_t *send, const int64_t *send_counts, const int64_t *send_offsets,
                      int64_t *recv, const int64_t *recv_counts, const int64_t *recv_offsets, void *stream);
/* the same for per-peer buffers that are separate allocations (host arrays [world] of device pointers / byte counts) */
int bns_alltoallv_bytes(bns_ctx_t *c, const void *const *send_ptrs, const int64_t *send_bytes, void *const *recv_ptrs,
                        const int64_t *recv_bytes, void *stream);

/* y = dropout_p(x) with the Philox mask of bns_ln_relu_dropout_fwd_f32 (counter = (row, vector, offset), key = seed):
 * module/model.py:80 for the layer-0 input; nothing but y is stored. */
int bns_dropout_f32(const float *x, int64_t ldx, int64_t n, int64_t F, float p, uint64_t seed, uint64_t offset,
                    const uint64_t *offset_dev, float *y, int64_t ldy, void *stream);
/* y[r, :] = x[r, :] * row_scale[r] + bias[:]      (row_scale / bias may be NULL: 1 / 0) */
int bns_scale_rows_f32(const float *x, int64_t ldx, int64_t n, int64_t F, const float *row_scale, const float *bias, float *y,
                       int64_t ldy, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* BNSGCN_H_ */
