// gat.cuh -- GATConv's attention as kernels (included by bnsgcn.cu).  Reference: module/model.py:96-132 builds
// dgl.nn.GATConv(in, out, heads, dropout, dropout); per layer DGL runs  e = leaky_relu(el_u + er_v)  (u_add_v),
// a = edge_softmax(e), a = attn_drop(a), rst_v = sum_u a_uv ft_u  (u_mul_e + sum) and their autograd.  Round 1 did the
// per-entry algebra with ~25 ATen launches over [nnz, heads] temporaries and one SpMM launch per head.  Here the
// algebra is staged: scalar row walks for the softmax, the tuned SpMM / SDDMM kernels for everything F-wide.
//
//   gat_proj_kernel / gat_proj_bwd_kernel   el = <ft, attn_l>, er = <ft, attn_r> per head and their backward
//   gat_scores_kernel        one warp per destination row, scalars only: score -> online max / sum -> probability P and
//                            dropped attention a' per entry (a' of the halo entries also at their compacted positions)
//   (rst = A' ft is the weighted SpMM per head: bns_spmm_weighted_f32 + bns_spmm_compact_f32;
//    d a' = <d rst_v, ft_u> is bns_sddmm_dot_f32)
//   gat_softmax_bwd_kernel   one warp per destination row, scalars only: d a' -> d e per entry (in place), d er_v
//   gat_colsum_kernel        d el_u = sum over the entries of column u of d e (walks the static transposes through their
//                            entry permutation: deterministic, no atomics)
//   (d ft = A'^T d rst is the weighted transposed SpMM: spmm_kernel with per-entry weights looked up through the
//    permutation, bns_spmm_weighted_f32)
//
// A fused form -- one warp per destination row doing scores, softmax, dropout and the weighted accumulation of the
// gathered ft rows in one launch per direction -- keeps one row's dependent loads in flight per warp; on a low-degree
// graph (Yelp shape, ~20 entries per row) that is a latency chain per row, and it measured 3x slower than the staged
// form, whose SpMM keeps 8 gathers in flight per lane (profiles/gat_r02.md).
//
// The row's entries are the inner ones (a_in) followed by this epoch's SAMPLED halo ones (a_out after
// bns_graph_compact_cols: chunk-local compaction, so a row is walked chunk by chunk through row_chunk).
namespace {

constexpr int kGatMaxHeads = 8;

struct GatGraph {
    const int64_t *in_ptr; const int32_t *in_idx;                          // a_in: CSR
    const int32_t *out_row_chunk; const int64_t *out_chunk_start;          // a_out: chunks of each row
    const int32_t *cidx, *chunk_cnt, *cpos;                                // its per-epoch compaction (NULL: no halo)
    int64_t n_rows, x_halo_base;
};

struct GatArgs {
    GatGraph g;
    int32_t H;
    const float *el, *er;                                                  // [n_u, H], [n_rows, H]
    float slope, p_drop, keep_scale;
    uint64_t seed, offset; const uint64_t *offset_dev;
    float *P_in, *P_out;                                                   // [nnz, H] at the ORIGINAL entry positions
    float *dE_in, *dE_out, *d_er;                                          // backward
};

__device__ __forceinline__ float leaky(float x, float slope) { return x > 0.f ? x : x * slope; }

// keep-mask of attention entry `gid` (a global entry id: inner entries first, then halo entries at their original
// positions), head h: one Philox4x32-10 call per (entry, 4 heads)
__device__ __forceinline__ bool gat_keep(uint64_t seed, uint64_t offset, int64_t gid, int h, float p) {
    uint32_t r[4];
    philox4x32_10((uint32_t)gid, (uint32_t)((uint64_t)gid >> 32) ^ 0x47415400u ^ (uint32_t)(h >> 2), (uint32_t)offset,
                  (uint32_t)(offset >> 32), (uint32_t)seed, (uint32_t)(seed >> 32), r);
    return (float)r[h & 3] * 2.3283064365386963e-10f >= p;
}

// Walks the entries of row v: f(position in the original CSR arrays, source row of ft, is_halo)
#define BNS_GAT_FOR_EACH_ENTRY(LANE_STRIDE_BODY)                                                     \
    for (int64_t k = a.g.in_ptr[v] + lane; k < a.g.in_ptr[v + 1]; k += 32) {                         \
        const int32_t u = a.g.in_idx[k];                                                             \
        const int64_t pos = k;                                                                       \
        const bool halo = false;                                                                     \
        LANE_STRIDE_BODY                                                                             \
    }                                                                                                \
    if (a.g.cidx) {                                                                                  \
        for (int32_t c = a.g.out_row_chunk[v]; c < a.g.out_row_chunk[v + 1]; ++c) {                  \
            const int64_t s0 = a.g.out_chunk_start[c];                                               \
            const int32_t cnt = a.g.chunk_cnt[c];                                                    \
            for (int32_t j = lane; j < cnt; j += 32) {                                               \
                const int32_t u = (int32_t)a.g.x_halo_base + a.g.cidx[s0 + j];                       \
                const int64_t pos = a.g.cpos[s0 + j];                                                \
                const bool halo = true;                                                              \
                LANE_STRIDE_BODY                                                                     \
            }                                                                                        \
        }                                                                                            \
    }

// P (probabilities, original positions), W (dropped attention a' = p * mask / (1 - q), original positions; may alias P
// when q == 0) and Wc (a' of the halo entries at their COMPACTED positions: the weights of bns_spmm_compact_f32)
__global__ void __launch_bounds__(kThreads) gat_scores_kernel(GatArgs a, int64_t nnz_in, float *W_in, float *W_out, float *Wc) {
    const int lane = threadIdx.x & 31;
    const int64_t warps_total = (int64_t)gridDim.x * kWarps;
    const uint64_t offset = a.offset + (a.offset_dev ? *a.offset_dev : 0ull);
    const int H = a.H;
    for (int64_t v = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); v < a.g.n_rows; v += warps_total) {
        float erv[kGatMaxHeads], m[kGatMaxHeads], l[kGatMaxHeads];
#pragma unroll
        for (int h = 0; h < kGatMaxHeads; ++h) {
            erv[h] = h < H ? a.er[v * H + h] : 0.f;
            m[h] = -INFINITY;
            l[h] = 0.f;
        }
        BNS_GAT_FOR_EACH_ENTRY({
            (void)pos; (void)halo;
_Pragma("unroll")
            for (int h = 0; h < kGatMaxHeads; ++h)
                if (h < H) {
                    const float sc = leaky(a.el[(int64_t)u * H + h] + erv[h], a.slope);
                    if (sc > m[h]) { l[h] = l[h] * expf(m[h] - sc) + 1.f; m[h] = sc; }
                    else l[h] += expf(sc - m[h]);
                }
        })
#pragma unroll
        for (int h = 0; h < kGatMaxHeads; ++h) {
            float mt = m[h];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) mt = fmaxf(mt, __shfl_xor_sync(0xffffffffu, mt, o));
            l[h] = warp_sum(m[h] == -INFINITY ? 0.f : l[h] * expf(m[h] - mt));
            m[h] = mt;
        }
        // second walk: probabilities and dropped attention
        for (int64_t k = a.g.in_ptr[v] + lane; k < a.g.in_ptr[v + 1]; k += 32) {
            const int32_t u = a.g.in_idx[k];
#pragma unroll
            for (int h = 0; h < kGatMaxHeads; ++h)
                if (h < H) {
                    const float p = expf(leaky(a.el[(int64_t)u * H + h] + erv[h], a.slope) - m[h]) / l[h];
                    a.P_in[k * H + h] = p;
                    if (a.p_drop > 0.f) W_in[k * H + h] = gat_keep(a.seed, offset, k, h, a.p_drop) ? p * a.keep_scale : 0.f;
                }
        }
        if (a.g.cidx) {
            for (int32_t c = a.g.out_row_chunk[v]; c < a.g.out_row_chunk[v + 1]; ++c) {
                const int64_t s0 = a.g.out_chunk_start[c];
                const int32_t cnt = a.g.chunk_cnt[c];
                for (int32_t j = lane; j < cnt; j += 32) {
                    const int32_t u = (int32_t)a.g.x_halo_base + a.g.cidx[s0 + j];
                    const int64_t pos = a.g.cpos[s0 + j];
#pragma unroll
                    for (int h = 0; h < kGatMaxHeads; ++h)
                        if (h < H) {
                            const float p = expf(leaky(a.el[(int64_t)u * H + h] + erv[h], a.slope) - m[h]) / l[h];
                            float wt = p;
                            if (a.p_drop > 0.f) wt = gat_keep(a.seed, offset, nnz_in + pos, h, a.p_drop) ? p * a.keep_scale : 0.f;
                            a.P_out[pos * H + h] = p;
                            if (a.p_drop > 0.f) W_out[pos * H + h] = wt;
                            Wc[(s0 + j) * H + h] = wt;
                        }
                }
            }
        }
    }
}

// in: dE_in / dE_out hold d a' (the SDDMM <d rst_v, ft_u>) at the original positions; out: d e in place, d er
__global__ void __launch_bounds__(kThreads) gat_softmax_bwd_kernel(GatArgs a, int64_t nnz_in) {
    const int lane = threadIdx.x & 31;
    const int64_t warps_total = (int64_t)gridDim.x * kWarps;
    const uint64_t offset = a.offset + (a.offset_dev ? *a.offset_dev : 0ull);
    const int H = a.H;
    for (int64_t v = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); v < a.g.n_rows; v += warps_total) {
        float erv[kGatMaxHeads], rowdot[kGatMaxHeads], der[kGatMaxHeads];
#pragma unroll
        for (int h = 0; h < kGatMaxHeads; ++h) {
            erv[h] = h < H ? a.er[v * H + h] : 0.f;
            rowdot[h] = 0.f;
            der[h] = 0.f;
        }
        BNS_GAT_FOR_EACH_ENTRY({
            (void)u;
            const float *P = (halo ? a.P_out : a.P_in) + pos * H;
            float *dE = (halo ? a.dE_out : a.dE_in) + pos * H;
            const int64_t gid = halo ? nnz_in + pos : pos;
_Pragma("unroll")
            for (int h = 0; h < kGatMaxHeads; ++h)
                if (h < H) {
                    float ms = 1.f;
                    if (a.p_drop > 0.f) ms = gat_keep(a.seed, offset, gid, h, a.p_drop) ? a.keep_scale : 0.f;
                    const float dp = dE[h] * ms;
                    dE[h] = dp;
                    rowdot[h] += P[h] * dp;
                }
        })
#pragma unroll
        for (int h = 0; h < kGatMaxHeads; ++h) rowdot[h] = warp_sum(rowdot[h]);
        BNS_GAT_FOR_EACH_ENTRY({
            const float *P = (halo ? a.P_out : a.P_in) + pos * H;
            float *dE = (halo ? a.dE_out : a.dE_in) + pos * H;
_Pragma("unroll")
            for (int h = 0; h < kGatMaxHeads; ++h)
                if (h < H) {
                    const float ds = P[h] * (dE[h] - rowdot[h]);
                    const float raw = a.el[(int64_t)u * H + h] + erv[h];
                    const float de = raw > 0.f ? ds : ds * a.slope;
                    dE[h] = de;
                    der[h] += de;
                }
        })
#pragma unroll
        for (int h = 0; h < kGatMaxHeads; ++h) {
            der[h] = warp_sum(der[h]);
            if (lane == 0 && h < H) a.d_er[v * H + h] = der[h];
        }
    }
}

// out[orow(r), h] = sum over the entries k of row r of the (transposed) graph of dE[perm[k], h]
__global__ void __launch_bounds__(kThreads) gat_colsum_kernel(const int64_t *__restrict__ indptr, const int32_t *__restrict__ perm,
                                                             int64_t n_rows, const float *__restrict__ dE, int32_t H,
                                                             const int32_t *__restrict__ row_map, int64_t out_base,
                                                             float *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warps_total = (int64_t)gridDim.x * kWarps;
    for (int64_t r = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); r < n_rows; r += warps_total) {
        int64_t orow = r;
        if (row_map) {
            const int32_t mrow = row_map[r];
            if (mrow < 0) continue;
            orow = mrow;
        }
        float acc[kGatMaxHeads];
#pragma unroll
        for (int h = 0; h < kGatMaxHeads; ++h) acc[h] = 0.f;
        for (int64_t k = indptr[r] + lane; k < indptr[r + 1]; k += 32) {
            const float *d = dE + (int64_t)perm[k] * H;
#pragma unroll
            for (int h = 0; h < kGatMaxHeads; ++h)
                if (h < H) acc[h] += d[h];
        }
#pragma unroll
        for (int h = 0; h < kGatMaxHeads; ++h) {
            acc[h] = warp_sum(acc[h]);
            if (lane == 0 && h < H) out[(out_base + orow) * H + h] = acc[h];
        }
    }
}


#undef BNS_GAT_FOR_EACH_ENTRY

int gat_fill(GatArgs &a, const bns_graph *a_in, const bns_graph *a_out, const int32_t *cidx, const int32_t *chunk_cnt,
             const int32_t *cpos, int64_t x_halo_base, const char *who) {
    BNS_REQUIRE(a_in, "%s: NULL inner graph", who);
    a.g.in_ptr = a_in->indptr; a.g.in_idx = a_in->indices; a.g.n_rows = a_in->n_rows; a.g.x_halo_base = x_halo_base;
    a.g.out_row_chunk = nullptr; a.g.out_chunk_start = nullptr; a.g.cidx = nullptr; a.g.chunk_cnt = nullptr; a.g.cpos = nullptr;
    if (a_out && cidx) {
        BNS_REQUIRE(chunk_cnt && cpos, "%s: the halo compaction needs chunk_cnt and cpos", who);
        BNS_REQUIRE(a_out->n_rows == a_in->n_rows, "%s: inner and halo matrices must have the same rows", who);
        a.g.out_row_chunk = a_out->row_chunk; a.g.out_chunk_start = a_out->chunk_start;
        a.g.cidx = cidx; a.g.chunk_cnt = chunk_cnt; a.g.cpos = cpos;
    }
    return BNS_OK;
}

inline unsigned gat_grid(int64_t n) {
    int64_t want = (n + kWarps - 1) / kWarps, cap = (int64_t)sm_count() * 6;
    return (unsigned)(want < cap ? (want > 0 ? want : 1) : cap);
}

}  // namespace

extern "C" int bns_gat_scores_f32(const bns_graph_t *a_in, const bns_graph_t *a_out, const int32_t *cidx, const int32_t *chunk_cnt,
                                  const int32_t *cpos, int64_t x_halo_base, int32_t H, const float *el, const float *er,
                                  float slope, float p_drop, uint64_t seed, uint64_t offset, const uint64_t *offset_dev,
                                  float *P_in, float *P_out, float *W_in, float *W_out, float *W_out_compact, void *stream) {
    GatArgs a{};
    int rc = gat_fill(a, a_in, a_out, cidx, chunk_cnt, cpos, x_halo_base, "bns_gat_scores_f32");
    if (rc) return rc;
    BNS_REQUIRE(H >= 1 && H <= kGatMaxHeads, "bns_gat_scores_f32: 1 <= heads <= 8");
    if (a.g.n_rows == 0) return BNS_OK;
    BNS_REQUIRE(el && er && P_in && (a.g.cidx == nullptr || (P_out && W_out_compact)), "bns_gat_scores_f32: NULL pointer");
    BNS_REQUIRE(p_drop >= 0.f && p_drop < 1.f, "bns_gat_scores_f32: p must be in [0, 1)");
    BNS_REQUIRE(p_drop == 0.f || (W_in && (a.g.cidx == nullptr || W_out)), "bns_gat_scores_f32: dropout needs W_in / W_out");
    a.H = H; a.el = el; a.er = er; a.slope = slope; a.p_drop = p_drop; a.keep_scale = 1.f / (1.f - p_drop);
    a.seed = seed; a.offset = offset; a.offset_dev = offset_dev; a.P_in = P_in; a.P_out = P_out;
    int64_t want = (a.g.n_rows + kWarps - 1) / kWarps, cap = (int64_t)sm_count() * 8;
    gat_scores_kernel<<<(unsigned)(want < cap ? want : cap), kThreads, 0, as_stream(stream)>>>(a, a_in->nnz, W_in, W_out, W_out_compact);
    ++g_launches;
    BNS_CUDA(cudaGetLastError());
    return BNS_OK;
}

extern "C" int bns_gat_softmax_bwd_f32(const bns_graph_t *a_in, const bns_graph_t *a_out, const int32_t *cidx,
                                       const int32_t *chunk_cnt, const int32_t *cpos, int64_t x_halo_base, int32_t H,
                                       const float *el, const float *er, float slope, float p_drop, uint64_t seed,
                                       uint64_t offset, const uint64_t *offset_dev, const float *P_in, const float *P_out,
                                       float *dE_in, float *dE_out, float *d_er, void *stream) {
    GatArgs a{};
    int rc = gat_fill(a, a_in, a_out, cidx, chunk_cnt, cpos, x_halo_base, "bns_gat_softmax_bwd_f32");
    if (rc) return rc;
    BNS_REQUIRE(H >= 1 && H <= kGatMaxHeads, "bns_gat_softmax_bwd_f32: 1 <= heads <= 8");
    if (a.g.n_rows == 0) return BNS_OK;
    BNS_REQUIRE(el && er && P_in && dE_in && d_er && (a.g.cidx == nullptr || (P_out && dE_out)), "bns_gat_softmax_bwd_f32: NULL pointer");
    a.H = H; a.el = el; a.er = er; a.slope = slope; a.p_drop = p_drop; a.keep_scale = 1.f / (1.f - p_drop);
    a.seed = seed; a.offset = offset; a.offset_dev = offset_dev;
    a.P_in = const_cast<float *>(P_in); a.P_out = const_cast<float *>(P_out); a.dE_in = dE_in; a.dE_out = dE_out; a.d_er = d_er;
    int64_t want = (a.g.n_rows + kWarps - 1) / kWarps, cap = (int64_t)sm_count() * 8;
    gat_softmax_bwd_kernel<<<(unsigned)(want < cap ? want : cap), kThreads, 0, as_stream(stream)>>>(a, a_in->nnz);
    ++g_launches;
    BNS_CUDA(cudaGetLastError());
    return BNS_OK;
}

// d_el[out_base + orow(r), :H] = sum over the entries of row r of the TRANSPOSED graph gT of dE[perm[k], :H]
extern "C" int bns_gat_colsum_f32(const bns_graph_t *gT, const float *dE, int32_t H, const int32_t *row_map, int64_t out_base,
                                  float *d_el, void *stream) {
    BNS_REQUIRE(gT && gT->perm, "bns_gat_colsum_f32: needs a graph made by bns_graph_transpose");
    BNS_REQUIRE(H >= 1 && H <= kGatMaxHeads, "bns_gat_colsum_f32: 1 <= heads <= 8");
    if (gT->n_rows == 0) return BNS_OK;
    BNS_REQUIRE(d_el && (dE || gT->nnz == 0), "bns_gat_colsum_f32: NULL pointer");
    gat_colsum_kernel<<<gat_grid(gT->n_rows), kThreads, 0, as_stream(stream)>>>(gT->indptr, gT->perm, gT->n_rows, dE, H, row_map,
                                                                               out_base, d_el);
    ++g_launches;
    BNS_CUDA(cudaGetLastError());
    return BNS_OK;
}

// ---- el = <ft, attn_l>, er = <ft, attn_r> per head (the two reductions of dgl.nn.GATConv before the edge scores) ------------
namespace {

// out[r, h] = < X[r, h*Fo : (h+1)*Fo], a[h, :] >; one warp per row
__global__ void __launch_bounds__(kThreads) gat_proj_kernel(const float *__restrict__ X, int64_t ldx, int64_t rows, int32_t H,
                                                           int32_t Fo, const float *__restrict__ a, float *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warps_total = (int64_t)gridDim.x * kWarps;
    const int cvh = Fo / 4;
    for (int64_t r = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); r < rows; r += warps_total) {
        const float4 *x = reinterpret_cast<const float4 *>(X + r * ldx);
        for (int h = 0; h < H; ++h) {
            float acc = 0.f;
            for (int c = h * cvh + lane; c < (h + 1) * cvh; c += 32) {
                const float4 v = __ldg(x + c), w = __ldg(reinterpret_cast<const float4 *>(a) + c);
                acc += (v.x * w.x + v.y * w.y) + (v.z * w.z + v.w * w.w);
            }
            acc = warp_sum(acc);
            if (lane == 0) out[r * H + h] = acc;
        }
    }
}

// dX[r, c] (+)= s[r, head(c)] * a[c];   partial[block, c] = sum over the block's rows of s[r, head(c)] * X[r, c]
// (thread (rg, c) owns float4 column c of every RG-th row of the block's row range: fixed order, like colsum2_partial_kernel)
__global__ void __launch_bounds__(kThreads) gat_proj_bwd_kernel(const float *__restrict__ X, int64_t ldx, int64_t rows, int32_t H,
                                                               int32_t Fo, int CV, const float4 *__restrict__ a,
                                                               const float *__restrict__ s, float *dX, int64_t lddx,
                                                               int accumulate, float4 *__restrict__ partial) {
    __shared__ float4 s0[kThreads];
    const int RG = kThreads / CV;
    const int rg = threadIdx.x / CV, c = threadIdx.x % CV;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (rg < RG) {
        const int hd = (c * 4) / Fo;
        const float4 av = a[c];
        const int64_t per = (rows + gridDim.x - 1) / gridDim.x;
        const int64_t r0 = (int64_t)blockIdx.x * per, r1 = r0 + per < rows ? r0 + per : rows;
        for (int64_t r = r0 + rg; r < r1; r += RG) {
            const float sv = __ldg(s + r * H + hd);
            const float4 x = __ldg(reinterpret_cast<const float4 *>(X + r * ldx) + c);
            acc.x = fmaf(sv, x.x, acc.x); acc.y = fmaf(sv, x.y, acc.y); acc.z = fmaf(sv, x.z, acc.z); acc.w = fmaf(sv, x.w, acc.w);
            float4 *d = reinterpret_cast<float4 *>(dX + r * lddx) + c;
            float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
            if (accumulate) o = *d;
            o.x = fmaf(sv, av.x, o.x); o.y = fmaf(sv, av.y, o.y); o.z = fmaf(sv, av.z, o.z); o.w = fmaf(sv, av.w, o.w);
            *d = o;
        }
    }
    s0[threadIdx.x] = acc;
    __syncthreads();
    if (rg == 0) {
        for (int g = 1; g < RG; ++g) {
            const float4 u = s0[g * CV + c];
            acc.x += u.x; acc.y += u.y; acc.z += u.z; acc.w += u.w;
        }
        partial[(int64_t)blockIdx.x * CV + c] = acc;
    }
}

}  // namespace

extern "C" int bns_gat_proj_f32(const float *X, int64_t ldx, int64_t rows, int32_t H, int32_t Fo, const float *attn, float *out,
                                void *stream) {
    BNS_REQUIRE(H >= 1 && Fo >= 4 && Fo % 4 == 0 && (int64_t)H * Fo <= kColsumMaxCols, "bns_gat_proj_f32: need Fo %% 4 == 0 and heads * Fo <= 1024");
    if (rows == 0) return BNS_OK;
    BNS_REQUIRE(X && attn && out && ldx % 4 == 0 && ldx >= (int64_t)H * Fo, "bns_gat_proj_f32: bad matrix");
    BNS_REQUIRE(((reinterpret_cast<uintptr_t>(X) | reinterpret_cast<uintptr_t>(attn)) & 15u) == 0, "bns_gat_proj_f32: unaligned");
    gat_proj_kernel<<<ln_grid(rows), kThreads, 0, as_stream(stream)>>>(X, ldx, rows, H, Fo, attn, out);
    ++g_launches;
    BNS_CUDA(cudaGetLastError());
    return BNS_OK;
}

// d X (+)= s (x) attn per head, d attn = sum_r s[r, h] X[r, h, :] (deterministic two-stage sum).  ws: bns_colsum_workspace_bytes(H * Fo)
extern "C" int bns_gat_proj_bwd_f32(const float *X, int64_t ldx, int64_t rows, int32_t H, int32_t Fo, const float *attn,
                                    const float *s, float *dX, int64_t lddx, int accumulate, float *d_attn, void *ws,
                                    size_t ws_bytes, void *stream) {
    const int64_t HF = (int64_t)H * Fo;
    BNS_REQUIRE(H >= 1 && Fo >= 4 && Fo % 4 == 0 && HF <= kColsumMaxCols, "bns_gat_proj_bwd_f32: need Fo %% 4 == 0 and heads * Fo <= 1024");
    BNS_REQUIRE(d_attn && attn, "bns_gat_proj_bwd_f32: NULL argument");
    cudaStream_t st = as_stream(stream);
    if (rows == 0) {
        BNS_CUDA(cudaMemsetAsync(d_attn, 0, (size_t)HF * sizeof(float), st));
        return BNS_OK;
    }
    BNS_REQUIRE(X && s && dX && ldx % 4 == 0 && lddx % 4 == 0 && ldx >= HF && lddx >= HF, "bns_gat_proj_bwd_f32: bad matrix");
    BNS_REQUIRE(((reinterpret_cast<uintptr_t>(X) | reinterpret_cast<uintptr_t>(attn) | reinterpret_cast<uintptr_t>(dX) |
                  reinterpret_cast<uintptr_t>(d_attn)) & 15u) == 0, "bns_gat_proj_bwd_f32: unaligned");
    if (!ws || ws_bytes < bns_colsum_workspace_bytes(HF) || (reinterpret_cast<uintptr_t>(ws) & 15u))
        return fail(BNS_E_WORKSPACE, "bns_gat_proj_bwd_f32: workspace %zu bytes < %zu needed", ws_bytes, bns_colsum_workspace_bytes(HF));
    const int CV = (int)(HF / 4);
    int blocks = colsum_blocks();
    if ((int64_t)blocks > rows) blocks = (int)rows;
    gat_proj_bwd_kernel<<<blocks, kThreads, 0, st>>>(X, ldx, rows, H, Fo, CV, reinterpret_cast<const float4 *>(attn), s, dX, lddx,
                                                     accumulate ? 1 : 0, reinterpret_cast<float4 *>(ws));
    colsum_final_kernel<<<(CV + kWarps - 1) / kWarps, kThreads, 0, st>>>(reinterpret_cast<const float4 *>(ws), blocks, CV,
                                                                         reinterpret_cast<float4 *>(d_attn), nullptr);
    g_launches += 2;
    BNS_CUDA(cudaGetLastError());
    return BNS_OK;
}
