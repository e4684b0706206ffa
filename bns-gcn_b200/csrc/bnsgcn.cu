// bnsgcn.cu -- sm_100a kernels + the C ABI of include/bnsgcn.h.
//
// Hot kernels (all HBM/L2-bound f32 gather / scatter work; no tensor-core shaped math here):
//   spmm_kernel        K1/K1b/K2  nnz-balanced CSR row-sum, one warp per chunk, 16 B/lane gathers
//   spmm_fixup_kernel  deterministic combine of rows longer than one chunk
//   gather / scatter   K3/K5      boundary pack and gradient scatter-add
//   philox_key / take  K6         counter-based exactly-k sampling (with cub radix sort)
//   p2p_put_rows       K3+C1      pack straight into the peer's receive slab over NVLink + flag
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 --shared -Xcompiler -fPIC
#include "bnsgcn.h"

#include <cuda_runtime.h>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <new>

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define BNS_CUDA(call)                                                                         \
    do {                                                                                       \
        cudaError_t e_ = (call);                                                               \
        if (e_ != cudaSuccess)                                                                 \
            return fail(BNS_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_),    \
                        __FILE__, __LINE__);                                                   \
    } while (0)

#define BNS_REQUIRE(cond, ...)                                                                 \
    do {                                                                                       \
        if (!(cond)) return fail(BNS_E_INVALID, __VA_ARGS__);                                  \
    } while (0)

inline cudaStream_t as_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kDefaultChunk = 256;   // B200 sweep (profiles/spmm_chunk_sweep_r1.txt): 256 -> 7.39 ms, 512 -> 7.58, 1024 -> 8.34, 2048 -> 9.27

std::atomic<unsigned long long> g_launches{0};   // kernels of this library enqueued so far (bench.py gpu_launches)

// Per-DEVICE properties (ranks that live as threads of one process may sit on different GPUs).
constexpr int kMaxDevices = 64;
struct DeviceProps {
    std::atomic<int> sms{0};
    std::atomic<long long> l2{0};
};
DeviceProps g_dev[kMaxDevices];

int current_device() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) dev = 0;
    return dev;
}

int sm_count() {
    const int dev = current_device();
    int n = g_dev[dev].sms.load(std::memory_order_relaxed);
    if (n == 0) {
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        g_dev[dev].sms.store(n, std::memory_order_relaxed);
    }
    return n;
}

}  // namespace

struct bns_graph {
    int64_t n_rows = 0, n_cols = 0, nnz = 0;
    int32_t chunk_nnz = 0;
    int64_t n_chunks = 0, n_split = 0, n_parts = 0;
    int64_t *indptr = nullptr;      // [n_rows+1]
    int32_t *indices = nullptr;     // [nnz]
    int32_t *chunk_row = nullptr;   // [n_chunks]
    int64_t *chunk_start = nullptr; // [n_chunks]
    int32_t *chunk_part = nullptr;  // [n_chunks]  partial-sum slot, -1 when the row is a single chunk
    int32_t *row_chunk = nullptr;   // [n_rows+1]  first chunk of each row (row r owns chunks row_chunk[r] .. row_chunk[r+1])
    int32_t *split_row = nullptr;   // [n_split]
    int32_t *split_part = nullptr;  // [n_split+1] first partial slot of each split row
    int32_t *perm = nullptr;        // transposes only: [nnz] entry k of this graph is entry perm[k] of its source
};

// =================================================================================================
// graph construction
// =================================================================================================
namespace {

__global__ void count_chunks_kernel(const int64_t *__restrict__ indptr, int64_t n_rows, int32_t chunk,
                                    int32_t *__restrict__ n_chunk, int32_t *__restrict__ n_part,
                                    int32_t *__restrict__ is_split) {
    int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    int64_t deg = indptr[r + 1] - indptr[r];
    int32_t c = deg <= chunk ? 1 : (int32_t)((deg + chunk - 1) / chunk);
    n_chunk[r] = c;
    n_part[r] = c > 1 ? c : 0;
    is_split[r] = c > 1 ? 1 : 0;
}

__global__ void fill_chunks_kernel(const int64_t *__restrict__ indptr, int64_t n_rows, int32_t chunk,
                                   const int32_t *__restrict__ chunk_off, const int32_t *__restrict__ part_off,
                                   const int32_t *__restrict__ split_off, int32_t *__restrict__ chunk_row,
                                   int64_t *__restrict__ chunk_start, int32_t *__restrict__ chunk_part,
                                   int32_t *__restrict__ split_row, int32_t *__restrict__ split_part) {
    int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    int32_t c0 = chunk_off[r], c1 = chunk_off[r + 1];
    int64_t s = indptr[r];
    bool split = (c1 - c0) > 1;
    int32_t p0 = part_off[r];
    for (int32_t c = c0; c < c1; ++c) {
        chunk_row[c] = (int32_t)r;
        chunk_start[c] = s + (int64_t)(c - c0) * chunk;
        chunk_part[c] = split ? p0 + (c - c0) : -1;
    }
    if (split) {
        int32_t i = split_off[r];
        split_row[i] = (int32_t)r;
        split_part[i] = p0;
    }
}

__global__ void set_last_kernel(int32_t *split_part, int64_t n_split, int32_t n_parts) {
    if (threadIdx.x == 0 && blockIdx.x == 0) split_part[n_split] = n_parts;
}

__global__ void expand_rows_kernel(const int64_t *__restrict__ indptr, int64_t n_rows, int32_t *__restrict__ rows) {
    // one warp per row
    int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (w >= n_rows) return;
    for (int64_t k = indptr[w] + lane; k < indptr[w + 1]; k += 32) rows[k] = (int32_t)w;
}

__global__ void lower_bound_kernel(const int32_t *__restrict__ sorted_keys, int64_t n, int64_t n_cols,
                                   int64_t *__restrict__ indptr) {
    int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (c > n_cols) return;
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        int64_t mid = (lo + hi) >> 1;
        if ((int64_t)sorted_keys[mid] < c) lo = mid + 1; else hi = mid;
    }
    indptr[c] = lo;
}

__global__ void iota_i32_kernel(int32_t *dst, int64_t n) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) dst[i] = (int32_t)i;
}

__global__ void gather_i32_kernel(const int32_t *__restrict__ src, const int32_t *__restrict__ idx, int64_t n,
                                  int32_t *__restrict__ dst) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[idx[i]];
}

__global__ void check_indices_kernel(const int32_t *__restrict__ idx, int64_t nnz, int64_t n_cols, int *bad) {
    int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k < nnz && (idx[k] < 0 || idx[k] >= n_cols)) *bad = 1;
}

int build_chunks(bns_graph *g, cudaStream_t st) {
    const int64_t n = g->n_rows;
    int32_t *n_chunk = nullptr, *n_part = nullptr, *is_split = nullptr;
    int32_t *chunk_off = nullptr, *part_off = nullptr, *split_off = nullptr;
    void *tmp = nullptr;
    size_t tmp_bytes = 0;
    BNS_CUDA(cudaMalloc(&n_chunk, (n + 1) * sizeof(int32_t)));
    BNS_CUDA(cudaMalloc(&n_part, (n + 1) * sizeof(int32_t)));
    BNS_CUDA(cudaMalloc(&is_split, (n + 1) * sizeof(int32_t)));
    BNS_CUDA(cudaMalloc(&chunk_off, (n + 1) * sizeof(int32_t)));
    BNS_CUDA(cudaMalloc(&part_off, (n + 1) * sizeof(int32_t)));
    BNS_CUDA(cudaMalloc(&split_off, (n + 1) * sizeof(int32_t)));
    BNS_CUDA(cudaMemsetAsync(n_chunk, 0, (n + 1) * sizeof(int32_t), st));
    BNS_CUDA(cudaMemsetAsync(n_part, 0, (n + 1) * sizeof(int32_t), st));
    BNS_CUDA(cudaMemsetAsync(is_split, 0, (n + 1) * sizeof(int32_t), st));
    if (n > 0) {
        count_chunks_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(g->indptr, n, g->chunk_nnz, n_chunk, n_part,
                                                                        is_split);
    }
    BNS_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, n_chunk, chunk_off, (int)(n + 1), st));
    BNS_CUDA(cudaMalloc(&tmp, tmp_bytes ? tmp_bytes : 16));
    BNS_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, n_chunk, chunk_off, (int)(n + 1), st));
    BNS_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, n_part, part_off, (int)(n + 1), st));
    BNS_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, is_split, split_off, (int)(n + 1), st));
    int32_t totals[3] = {0, 0, 0};
    BNS_CUDA(cudaMemcpyAsync(&totals[0], chunk_off + n, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    BNS_CUDA(cudaMemcpyAsync(&totals[1], part_off + n, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    BNS_CUDA(cudaMemcpyAsync(&totals[2], split_off + n, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    BNS_CUDA(cudaStreamSynchronize(st));
    g->n_chunks = totals[0];
    g->n_parts = totals[1];
    g->n_split = totals[2];
    BNS_CUDA(cudaMalloc(&g->chunk_row, (g->n_chunks + 1) * sizeof(int32_t)));
    BNS_CUDA(cudaMalloc(&g->chunk_start, (g->n_chunks + 1) * sizeof(int64_t)));
    BNS_CUDA(cudaMalloc(&g->chunk_part, (g->n_chunks + 1) * sizeof(int32_t)));
    BNS_CUDA(cudaMalloc(&g->split_row, (g->n_split + 1) * sizeof(int32_t)));
    BNS_CUDA(cudaMalloc(&g->split_part, (g->n_split + 2) * sizeof(int32_t)));
    if (n > 0) {
        fill_chunks_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(g->indptr, n, g->chunk_nnz, chunk_off, part_off,
                                                                       split_off, g->chunk_row, g->chunk_start,
                                                                       g->chunk_part, g->split_row, g->split_part);
    }
    set_last_kernel<<<1, 32, 0, st>>>(g->split_part, g->n_split, (int32_t)g->n_parts);
    BNS_CUDA(cudaGetLastError());
    BNS_CUDA(cudaStreamSynchronize(st));
    cudaFree(n_chunk); cudaFree(n_part); cudaFree(is_split);
    g->row_chunk = chunk_off;            // kept: the row-wise walkers (gat.cuh) go from a row to its chunks
    cudaFree(part_off); cudaFree(split_off); cudaFree(tmp);
    return BNS_OK;
}

}  // namespace

extern "C" int bns_abi_version(void) { return BNS_ABI_VERSION; }
extern "C" uint64_t bns_launch_count(void) { return g_launches.load(); }
extern "C" const char *bns_last_error(void) { return g_err; }

extern "C" int bns_device_info(char *name, size_t name_len, int *sms, int64_t *l2_bytes, int *cc_major, int *cc_minor) {
    int dev = 0;
    BNS_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    BNS_CUDA(cudaGetDeviceProperties(&prop, dev));
    if (name && name_len) {
        strncpy(name, prop.name, name_len - 1);
        name[name_len - 1] = 0;
    }
    if (sms) *sms = prop.multiProcessorCount;
    if (l2_bytes) *l2_bytes = prop.l2CacheSize;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    return BNS_OK;
}

extern "C" int bns_graph_destroy(bns_graph_t *g) {
    if (!g) return BNS_OK;
    cudaFree(g->indptr); cudaFree(g->indices); cudaFree(g->chunk_row); cudaFree(g->chunk_start);
    cudaFree(g->chunk_part); cudaFree(g->row_chunk); cudaFree(g->split_row); cudaFree(g->split_part); cudaFree(g->perm);
    delete g;
    return BNS_OK;
}

extern "C" int bns_graph_create(bns_graph_t **out, int64_t n_rows, int64_t n_cols, int64_t nnz,
                                const int64_t *indptr, const int32_t *indices, int32_t chunk_nnz, void *stream) {
    BNS_REQUIRE(out != nullptr, "bns_graph_create: out is NULL");
    BNS_REQUIRE(n_rows >= 0 && n_cols >= 0 && nnz >= 0, "bns_graph_create: negative size");
    BNS_REQUIRE(n_rows < INT32_MAX && n_cols < INT32_MAX, "bns_graph_create: more than 2^31-1 rows/cols");
    BNS_REQUIRE(indptr != nullptr, "bns_graph_create: indptr is NULL");
    BNS_REQUIRE(nnz == 0 || indices != nullptr, "bns_graph_create: indices is NULL");
    BNS_REQUIRE(chunk_nnz >= 0, "bns_graph_create: negative chunk_nnz");
    cudaStream_t st = as_stream(stream);
    bns_graph *g = new (std::nothrow) bns_graph();
    if (!g) return fail(BNS_E_INVALID, "bns_graph_create: out of host memory");
    g->n_rows = n_rows; g->n_cols = n_cols; g->nnz = nnz;
    g->chunk_nnz = chunk_nnz ? ((chunk_nnz + 31) / 32) * 32 : kDefaultChunk;
    int rc = BNS_OK;
    do {
        if (cudaMalloc(&g->indptr, (n_rows + 1) * sizeof(int64_t)) != cudaSuccess ||
            cudaMalloc(&g->indices, (nnz + 4) * sizeof(int32_t)) != cudaSuccess) {
            rc = fail(BNS_E_CUDA, "bns_graph_create: cudaMalloc failed: %s", cudaGetErrorString(cudaGetLastError()));
            break;
        }
        if (cudaMemcpyAsync(g->indptr, indptr, (n_rows + 1) * sizeof(int64_t), cudaMemcpyDeviceToDevice, st) != cudaSuccess ||
            (nnz && cudaMemcpyAsync(g->indices, indices, nnz * sizeof(int32_t), cudaMemcpyDeviceToDevice, st) != cudaSuccess)) {
            rc = fail(BNS_E_CUDA, "bns_graph_create: copy failed: %s", cudaGetErrorString(cudaGetLastError()));
            break;
        }
        // validate: indptr[0] == 0, indptr[n_rows] == nnz, indices in range
        int64_t ends[2] = {0, 0};
        cudaMemcpyAsync(&ends[0], g->indptr, sizeof(int64_t), cudaMemcpyDeviceToHost, st);
        cudaMemcpyAsync(&ends[1], g->indptr + n_rows, sizeof(int64_t), cudaMemcpyDeviceToHost, st);
        int *bad = nullptr, hbad = 0;
        if (cudaMalloc(&bad, sizeof(int)) != cudaSuccess) {
            rc = fail(BNS_E_CUDA, "bns_graph_create: cudaMalloc failed: %s", cudaGetErrorString(cudaGetLastError()));
            break;
        }
        cudaMemsetAsync(bad, 0, sizeof(int), st);
        if (nnz) check_indices_kernel<<<(unsigned)((nnz + 255) / 256), 256, 0, st>>>(g->indices, nnz, n_cols, bad);
        cudaMemcpyAsync(&hbad, bad, sizeof(int), cudaMemcpyDeviceToHost, st);
        cudaError_t e = cudaStreamSynchronize(st);
        cudaFree(bad);
        if (e != cudaSuccess) { rc = fail(BNS_E_CUDA, "bns_graph_create: %s", cudaGetErrorString(e)); break; }
        if (ends[0] != 0 || ends[1] != nnz) {
            rc = fail(BNS_E_INVALID, "bns_graph_create: indptr[0]=%lld indptr[n_rows]=%lld but nnz=%lld",
                      (long long)ends[0], (long long)ends[1], (long long)nnz);
            break;
        }
        if (hbad) { rc = fail(BNS_E_INVALID, "bns_graph_create: a column index is outside [0, n_cols)"); break; }
        rc = build_chunks(g, st);
    } while (0);
    if (rc != BNS_OK) { bns_graph_destroy(g); return rc; }
    *out = g;
    return BNS_OK;
}

extern "C" int bns_graph_transpose(const bns_graph_t *g, bns_graph_t **out, void *stream) {
    BNS_REQUIRE(g && out, "bns_graph_transpose: NULL argument");
    cudaStream_t st = as_stream(stream);
    const int64_t nnz = g->nnz;
    BNS_REQUIRE(nnz < INT32_MAX, "bns_graph_transpose: nnz >= 2^31 not supported by the sort");
    int32_t *rows = nullptr, *keys_out = nullptr, *vals_out = nullptr;
    int64_t *t_indptr = nullptr;
    void *tmp = nullptr;
    size_t tmp_bytes = 0;
    BNS_CUDA(cudaMalloc(&rows, (nnz + 1) * sizeof(int32_t)));
    BNS_CUDA(cudaMalloc(&keys_out, (nnz + 1) * sizeof(int32_t)));
    BNS_CUDA(cudaMalloc(&vals_out, (nnz + 1) * sizeof(int32_t)));
    BNS_CUDA(cudaMalloc(&t_indptr, (g->n_cols + 1) * sizeof(int64_t)));
    if (g->n_rows > 0) {
        int64_t threads = g->n_rows * 32;
        expand_rows_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(g->indptr, g->n_rows, rows);
    }
    int32_t *eid = nullptr, *perm = nullptr;
    BNS_CUDA(cudaMalloc(&eid, (nnz + 1) * sizeof(int32_t)));
    BNS_CUDA(cudaMalloc(&perm, (nnz + 1) * sizeof(int32_t)));
    if (nnz > 0) iota_i32_kernel<<<(unsigned)((nnz + 255) / 256), 256, 0, st>>>(eid, nnz);
    int end_bit = 1;
    while (end_bit < 32 && ((int64_t)1 << end_bit) < g->n_cols) ++end_bit;
    // stable sort of the entries by column: values = entry ids, so the permutation survives (per-entry weights of
    // the source graph -- GAT attention -- are carried to the transpose with it)
    BNS_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, g->indices, keys_out, eid, perm, (int)nnz, 0,
                                             end_bit, st));
    BNS_CUDA(cudaMalloc(&tmp, tmp_bytes ? tmp_bytes : 16));
    BNS_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, g->indices, keys_out, eid, perm, (int)nnz, 0,
                                             end_bit, st));
    if (nnz > 0) gather_i32_kernel<<<(unsigned)((nnz + 255) / 256), 256, 0, st>>>(rows, perm, nnz, vals_out);
    lower_bound_kernel<<<(unsigned)((g->n_cols + 1 + 255) / 256), 256, 0, st>>>(keys_out, nnz, g->n_cols, t_indptr);
    BNS_CUDA(cudaGetLastError());
    BNS_CUDA(cudaStreamSynchronize(st));
    int rc = bns_graph_create(out, g->n_cols, g->n_rows, nnz, t_indptr, vals_out, g->chunk_nnz, stream);
    if (rc == BNS_OK) (*out)->perm = perm; else cudaFree(perm);
    cudaFree(rows); cudaFree(keys_out); cudaFree(vals_out); cudaFree(t_indptr); cudaFree(tmp); cudaFree(eid);
    return rc;
}

extern "C" int bns_graph_copy_perm(const bns_graph_t *g, int32_t *perm_out, void *stream) {
    BNS_REQUIRE(g && perm_out, "bns_graph_copy_perm: NULL argument");
    BNS_REQUIRE(g->perm != nullptr, "bns_graph_copy_perm: not a graph made by bns_graph_transpose");
    if (g->nnz)
        BNS_CUDA(cudaMemcpyAsync(perm_out, g->perm, g->nnz * sizeof(int32_t), cudaMemcpyDeviceToDevice, as_stream(stream)));
    return BNS_OK;
}

extern "C" int bns_graph_info(const bns_graph_t *g, int64_t *n_rows, int64_t *n_cols, int64_t *nnz,
                              int64_t *n_chunks, int64_t *n_split_rows) {
    BNS_REQUIRE(g, "bns_graph_info: NULL graph");
    if (n_rows) *n_rows = g->n_rows;
    if (n_cols) *n_cols = g->n_cols;
    if (nnz) *nnz = g->nnz;
    if (n_chunks) *n_chunks = g->n_chunks;
    if (n_split_rows) *n_split_rows = g->n_split;
    return BNS_OK;
}

extern "C" int bns_graph_copy_csr(const bns_graph_t *g, int64_t *indptr_out, int32_t *indices_out, void *stream) {
    BNS_REQUIRE(g, "bns_graph_copy_csr: NULL graph");
    cudaStream_t st = as_stream(stream);
    if (indptr_out)
        BNS_CUDA(cudaMemcpyAsync(indptr_out, g->indptr, (g->n_rows + 1) * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
    if (indices_out && g->nnz)
        BNS_CUDA(cudaMemcpyAsync(indices_out, g->indices, g->nnz * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
    return BNS_OK;
}

// =================================================================================================
// SpMM
// =================================================================================================
namespace {

struct SpmmArgs {
    const int64_t *indptr;
    const int32_t *indices;
    const int32_t *chunk_row;
    const int64_t *chunk_start;
    const int32_t *chunk_part;
    const int32_t *chunk_cnt;      // compact mode (bns_graph_compact_cols): live entries of each chunk, NULL otherwise
    const int32_t *split_row;
    const int32_t *split_part;
    int64_t n_chunks, n_split;
    int32_t chunk_nnz;
    const float *X;
    int64_t ldx;
    float *Y;
    int64_t ldy;
    int32_t F;
    const float *row_scale;
    const float *col_scale;
    const float *edge_weight;   // per entry (CSR order) or NULL
    const int32_t *edge_perm;   // optional: entry k's weight is edge_weight[edge_perm[k] * edge_ld] (weights kept in the
    int64_t edge_ld;            // ORDER OF ANOTHER GRAPH, e.g. the source graph of a transpose; [nnz, heads] layouts)
    const int32_t *row_map;
    const int32_t *col_map;
    int32_t n_direct;
    int32_t accumulate;
    float *ws;
    int64_t ldws;
    int64_t n_tiles;     // column slabs of the kernel's SLAB width covering F
};

template <int W> struct Vec;
template <> struct Vec<4> {
    float4 v;
    __device__ __forceinline__ void zero() { v = make_float4(0.f, 0.f, 0.f, 0.f); }
    __device__ __forceinline__ void load_ro(const float *p) { v = __ldg(reinterpret_cast<const float4 *>(p)); }
    __device__ __forceinline__ void load(const float *p) { v = *reinterpret_cast<const float4 *>(p); }
    __device__ __forceinline__ void store(float *p) const { *reinterpret_cast<float4 *>(p) = v; }
    __device__ __forceinline__ void add(const Vec &o) { v.x += o.v.x; v.y += o.v.y; v.z += o.v.z; v.w += o.v.w; }
    __device__ __forceinline__ void fma(const Vec &o, float s) {
        v.x = fmaf(o.v.x, s, v.x); v.y = fmaf(o.v.y, s, v.y); v.z = fmaf(o.v.z, s, v.z); v.w = fmaf(o.v.w, s, v.w);
    }
    __device__ __forceinline__ void scale(float s) { v.x *= s; v.y *= s; v.z *= s; v.w *= s; }
    __device__ __forceinline__ void add_shfl_xor(int off) {
        v.x += __shfl_xor_sync(0xffffffffu, v.x, off); v.y += __shfl_xor_sync(0xffffffffu, v.y, off);
        v.z += __shfl_xor_sync(0xffffffffu, v.z, off); v.w += __shfl_xor_sync(0xffffffffu, v.w, off);
    }
};
template <> struct Vec<1> {
    float v;
    __device__ __forceinline__ void zero() { v = 0.f; }
    __device__ __forceinline__ void load_ro(const float *p) { v = __ldg(p); }
    __device__ __forceinline__ void load(const float *p) { v = *p; }
    __device__ __forceinline__ void store(float *p) const { *p = v; }
    __device__ __forceinline__ void add(const Vec &o) { v += o.v; }
    __device__ __forceinline__ void fma(const Vec &o, float s) { v = fmaf(o.v, s, v); }
    __device__ __forceinline__ void scale(float s) { v *= s; }
    __device__ __forceinline__ void add_shfl_xor(int off) { v += __shfl_xor_sync(0xffffffffu, v, off); }
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ int32_t ld_stream_i32(const int32_t *p) {
    int32_t r;
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}

// One warp per chunk of <= chunk_nnz entries of one row.  Lane l owns columns
//   f0 + (l + 32 t) * W .. + W   for t < NV   (W = 4: one 16-byte vector, W = 1: scalar path)
// so a warp reads each gathered row as NV fully coalesced 512-byte (W=4) requests.
// Column ids of 32 entries are fetched with one coalesced load, mapped (col_map: sampled halo ->
// slab row, -1 = skip), compacted through shared memory and then consumed UNROLL at a time so that
// UNROLL*NV independent 16-byte gathers are in flight per lane.
//
// Cache blocking (the ncu capture of round 1 showed why: with the whole F = 256 row per gather the 238 MB
// source matrix of the Reddit-shape graph misses the 126 MB L2 58 % of the time and the kernel moves 53 GB
// of DRAM per launch for 0.9 GB of algorithmic bytes).  The feature dimension is cut into column slabs of
// SLAB = G*W*NV floats chosen so that (source rows x SLAB x 4 B) stays L2-resident; work items are ordered
// slab-major, so at any moment all resident warps gather from the same slab.  For narrow slabs a warp is
// split into 32/G row groups of G lanes that walk different entries of the chunk concurrently (every lane
// still issues 16-byte loads) and are summed with shuffles at the end.
template <int W, int G, int NV, bool MAP, bool CSCALE, bool GUARD>
__global__ void __launch_bounds__(kThreads, (NV <= 1 ? 5 : 4)) spmm_kernel(SpmmArgs a) {
    constexpr int NG = 32 / G;                               // entries walked concurrently by one warp
    constexpr int UNROLL = (NV <= 2) ? 8 / NV : 2;           // independent 16-byte gathers in flight per lane
    constexpr int SLAB = G * W * NV;
    __shared__ int32_t s_col[kWarps][32];
    __shared__ float s_sc[kWarps][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int gi = lane / G, gl = lane % G;
    const int64_t warps_total = (int64_t)gridDim.x * kWarps;
    const int64_t items = a.n_chunks * a.n_tiles;
    for (int64_t item = (int64_t)blockIdx.x * kWarps + w; item < items; item += warps_total) {
        const int64_t c = item % a.n_chunks;
        const int f0 = (int)(item / a.n_chunks) * SLAB;
        int fcol[NV];
        bool fok[NV];
#pragma unroll
        for (int t = 0; t < NV; ++t) {
            fcol[t] = f0 + (gl + G * t) * W;
            fok[t] = !GUARD || fcol[t] < a.F;
        }
        const int32_t row = a.chunk_row[c];
        int32_t orow = row;
        if (a.row_map) {
            orow = a.row_map[row];
            if (orow < 0) continue;
        }
        const int64_t s = a.chunk_start[c];
        int64_t e;
        if (a.chunk_cnt) {         // per-epoch compacted indices: the chunk's live entries sit at the start of its range
            const int32_t cnt = a.chunk_cnt[c];
            // nothing sampled in this chunk: adding zero to Y would only cost a read-modify-write of the row
            if (cnt == 0 && a.accumulate && a.chunk_part[c] < 0) continue;
            e = s + cnt;
        } else {
            e = a.indptr[row + 1];
            if (e > s + a.chunk_nnz) e = s + a.chunk_nnz;
        }
        Vec<W> acc[NV];
#pragma unroll
        for (int t = 0; t < NV; ++t) acc[t].zero();
        for (int64_t k0 = s; k0 < e; k0 += 32) {
            const int64_t k = k0 + lane;
            int32_t col = -1;
            float sc = 1.f;
            if (k < e) {
                col = ld_stream_i32(a.indices + k);
                if (CSCALE) {        // per-source and / or per-entry weight (GAT attention) -> the FMA path
                    if (a.col_scale) sc = __ldg(a.col_scale + col);
                    if (a.edge_weight) sc *= __ldg(a.edge_weight + (a.edge_perm ? (int64_t)__ldg(a.edge_perm + k) : k) * a.edge_ld);
                }
                if (MAP) {
                    if (col >= a.n_direct) col = __ldg(a.col_map + (col - a.n_direct));
                }
            }
            int cnt;
            if (MAP) {
                const unsigned m = __ballot_sync(0xffffffffu, col >= 0);
                cnt = __popc(m);
                if (col >= 0) {
                    const int pos = __popc(m & ((1u << lane) - 1u));
                    s_col[w][pos] = col;
                    if (CSCALE) s_sc[w][pos] = sc;
                }
            } else {
                const int64_t rem = e - k0;
                cnt = rem < 32 ? (int)rem : 32;
                s_col[w][lane] = col;
                if (CSCALE) s_sc[w][lane] = sc;
            }
            __syncwarp();
            int j = 0;
            for (; j + NG * UNROLL <= cnt; j += NG * UNROLL) {       // full steps: no predication
                Vec<W> v[UNROLL][NV];
#pragma unroll
                for (int u = 0; u < UNROLL; ++u) {
                    const float *xr = a.X + (int64_t)s_col[w][j + u * NG + gi] * a.ldx;
#pragma unroll
                    for (int t = 0; t < NV; ++t) {
                        if (fok[t]) v[u][t].load_ro(xr + fcol[t]); else v[u][t].zero();
                    }
                }
#pragma unroll
                for (int u = 0; u < UNROLL; ++u) {
                    const float cs = CSCALE ? s_sc[w][j + u * NG + gi] : 1.f;
#pragma unroll
                    for (int t = 0; t < NV; ++t) {
                        if (CSCALE) acc[t].fma(v[u][t], cs); else acc[t].add(v[u][t]);
                    }
                }
            }
            for (; j < cnt; j += NG) {                               // tail: one entry per row group
                const int jj = j + gi;
                if (jj < cnt) {
                    const float *xr = a.X + (int64_t)s_col[w][jj] * a.ldx;
                    const float cs = CSCALE ? s_sc[w][jj] : 1.f;
#pragma unroll
                    for (int t = 0; t < NV; ++t) {
                        if (fok[t]) {
                            Vec<W> v;
                            v.load_ro(xr + fcol[t]);
                            if (CSCALE) acc[t].fma(v, cs); else acc[t].add(v);
                        }
                    }
                }
            }
            __syncwarp();
        }
        if (NG > 1) {            // fold the row groups: afterwards group 0 (lanes < G) holds the chunk's sum
#pragma unroll
            for (int t = 0; t < NV; ++t)
#pragma unroll
                for (int off = 16; off >= G; off >>= 1) acc[t].add_shfl_xor(off);
            if (gi != 0) continue;
        }
        const int32_t part = a.chunk_part[c];
        if (part >= 0) {   // the row spans several chunks: park the raw partial sum, combined later
            float *wr = a.ws + (int64_t)part * a.ldws;
#pragma unroll
            for (int t = 0; t < NV; ++t)
                if (fok[t]) acc[t].store(wr + fcol[t]);
        } else {
            const float rs = a.row_scale ? a.row_scale[row] : 1.f;
            float *yr = a.Y + (int64_t)orow * a.ldy;
#pragma unroll
            for (int t = 0; t < NV; ++t) {
                if (!fok[t]) continue;
                if (a.row_scale) acc[t].scale(rs);
                if (a.accumulate) {
                    Vec<W> old;
                    old.load(yr + fcol[t]);
                    acc[t].add(old);
                }
                acc[t].store(yr + fcol[t]);
            }
        }
    }
}

// Rows longer than one chunk: add their partial sums in chunk order (deterministic), then finish
// exactly like the single-chunk epilogue.
template <int W, int NV, bool GUARD>
__global__ void __launch_bounds__(kThreads) spmm_fixup_kernel(SpmmArgs a) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int f0 = blockIdx.y * (32 * W * NV);
    const int64_t i = (int64_t)blockIdx.x * kWarps + w;
    if (i >= a.n_split) return;
    const int32_t row = a.split_row[i];
    int32_t orow = row;
    if (a.row_map) {
        orow = a.row_map[row];
        if (orow < 0) return;
    }
    const int32_t p0 = a.split_part[i], p1 = a.split_part[i + 1];
    const float rs = a.row_scale ? a.row_scale[row] : 1.f;
    float *yr = a.Y + (int64_t)orow * a.ldy;
#pragma unroll
    for (int t = 0; t < NV; ++t) {
        const int fc = f0 + (lane + 32 * t) * W;
        if (GUARD && fc >= a.F) continue;
        Vec<W> acc;
        acc.zero();
        for (int32_t p = p0; p < p1; ++p) {
            Vec<W> v;
            v.load(a.ws + (int64_t)p * a.ldws + fc);
            acc.add(v);
        }
        if (a.row_scale) acc.scale(rs);
        if (a.accumulate) {
            Vec<W> old;
            old.load(yr + fc);
            acc.add(old);
        }
        acc.store(yr + fc);
    }
}

template <int W, int G, int NV, bool MAP, bool CSCALE, bool GUARD>
int launch_spmm(SpmmArgs a, cudaStream_t st) {
    static std::atomic<int> occ[kMaxDevices];            // per device, per instantiation
    const int dev = current_device();
    int blocks_per_sm = occ[dev].load(std::memory_order_relaxed);
    if (blocks_per_sm == 0) {
        int n = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, spmm_kernel<W, G, NV, MAP, CSCALE, GUARD>, kThreads, 0) !=
                cudaSuccess || n < 1)
            n = 2;
        blocks_per_sm = n;
        occ[dev].store(n, std::memory_order_relaxed);
    }
    constexpr int SLAB = G * W * NV;
    a.n_tiles = (a.F + SLAB - 1) / SLAB;
    const int64_t items = a.n_chunks * a.n_tiles;
    int64_t want = (items + kWarps - 1) / kWarps;
    int64_t cap = (int64_t)sm_count() * blocks_per_sm;
    unsigned gx = (unsigned)(want < cap ? (want > 0 ? want : 1) : cap);
    spmm_kernel<W, G, NV, MAP, CSCALE, GUARD><<<gx, kThreads, 0, st>>>(a);
    g_launches += a.n_split > 0 ? 2 : 1;
    if (a.n_split > 0) {
        unsigned fx = (unsigned)((a.n_split + kWarps - 1) / kWarps);
        if (W == 4) {
            const int tiles = (a.F + 255) / 256;
            spmm_fixup_kernel<4, 2, true><<<dim3(fx, tiles), kThreads, 0, st>>>(a);
        } else {
            const int tiles = (a.F + 255) / 256;
            spmm_fixup_kernel<1, 8, true><<<dim3(fx, tiles), kThreads, 0, st>>>(a);
        }
    }
    return BNS_OK;
}

template <int W, int G, int NV>
int dispatch_flags(const SpmmArgs &a, cudaStream_t st) {
    const bool map = a.col_map != nullptr, cs = a.col_scale != nullptr || a.edge_weight != nullptr;
    const bool guard = (a.F % (G * W * NV)) != 0;
    if (guard) {
        if (map && cs) return launch_spmm<W, G, NV, true, true, true>(a, st);
        if (map) return launch_spmm<W, G, NV, true, false, true>(a, st);
        if (cs) return launch_spmm<W, G, NV, false, true, true>(a, st);
        return launch_spmm<W, G, NV, false, false, true>(a, st);
    }
    if (map && cs) return launch_spmm<W, G, NV, true, true, false>(a, st);
    if (map) return launch_spmm<W, G, NV, true, false, false>(a, st);
    if (cs) return launch_spmm<W, G, NV, false, true, false>(a, st);
    return launch_spmm<W, G, NV, false, false, false>(a, st);
}

inline int64_t ws_ld(int64_t F) { return (F + 3) / 4 * 4; }

int64_t l2_bytes() {
    const int dev = current_device();
    long long v = g_dev[dev].l2.load(std::memory_order_relaxed);
    if (v == 0) {
        int b = 0;
        v = (cudaDeviceGetAttribute(&b, cudaDevAttrL2CacheSize, dev) == cudaSuccess && b > 0) ? b : (126ll << 20);
        g_dev[dev].l2.store(v, std::memory_order_relaxed);
    }
    return v;
}

// Widest column slab (in floats: 256, 128, 64 or 32) whose source slab  x_rows * slab * 4 B  fits the L2 budget.
int pick_slab(int64_t F, int64_t x_rows, int32_t forced) {
    if (forced == 256 || forced == 128 || forced == 64 || forced == 32) return forced;
    const char *env = getenv("BNS_SPMM_SLAB");
    if (env) {
        int v = atoi(env);
        if (v == 256 || v == 128 || v == 64 || v == 32) return v;
    }
    // Measured on B200 (profiles/spmm_slab_sweep_r1.md, Reddit-shape, F = 256, 238 MB of sources): slab 256 ->
    // 10.2 ms, 128 -> 8.1 ms, 64 -> 8.5 ms, 32 -> 14.1 ms; a 51 MB source matrix is fastest unblocked.  So: full
    // rows while they fit comfortably, else 128 floats (a slab about the size of L2 still wins: the slab-major
    // order keeps the hot part resident and halves the index re-reads of 64), else 64; never 32.  When even a
    // 64-float slab cannot be L2-resident the gather is a pure HBM stream and the widest slab is best.
    const double l2 = (double)l2_bytes(), bytes_per_col = (double)x_rows * 4.0;
    const int fmax = F >= 256 ? 256 : (F > 64 ? 128 : 64);
    if (fmax >= 256 && bytes_per_col * 256.0 <= 0.55 * l2) return 256;
    if (fmax >= 128 && bytes_per_col * 128.0 <= 1.0 * l2) return 128;
    if (bytes_per_col * 64.0 <= 1.0 * l2) return 64;
    return fmax;
}

int spmm_dispatch(const SpmmArgs &a, int64_t x_rows, int32_t slab_hint, cudaStream_t st) {
    const int64_t F = a.F;
    const bool vec = (F % 4 == 0) && (a.ldx % 4 == 0) && (a.ldy % 4 == 0) &&
                     ((reinterpret_cast<uintptr_t>(a.X) | reinterpret_cast<uintptr_t>(a.Y)) % 16 == 0);
    if (vec) {
        int slab = pick_slab(F, x_rows, slab_hint);
        while (slab > 32 && slab / 2 >= F) slab >>= 1;       // never wider than needed (F = 64 -> 64-wide groups)
        switch (slab) {
            case 256: dispatch_flags<4, 32, 2>(a, st); break;
            case 128: dispatch_flags<4, 32, 1>(a, st); break;
            case 64:  dispatch_flags<4, 16, 1>(a, st); break;
            default:  dispatch_flags<4, 8, 1>(a, st); break;
        }
    } else {
        dispatch_flags<1, 32, 8>(a, st);
    }
    BNS_CUDA(cudaGetLastError());
    return BNS_OK;
}

}  // namespace

extern "C" size_t bns_spmm_workspace_bytes(const bns_graph_t *g, int64_t F) {
    if (!g || F <= 0) return 0;
    return (size_t)g->n_parts * (size_t)ws_ld(F) * sizeof(float);
}

extern "C" int bns_spmm_sum_f32(const bns_graph_t *g, const float *X, int64_t ldx, int64_t F, float *Y, int64_t ldy,
                                const float *row_scale, const float *col_scale, const float *edge_weight,
                                const int32_t *row_map, const int32_t *col_map, int64_t n_direct, int64_t x_rows,
                                int32_t slab_hint, int accumulate, void *ws, size_t ws_bytes, void *stream) {
    BNS_REQUIRE(g, "bns_spmm_sum_f32: NULL graph");
    BNS_REQUIRE(F > 0 && F < (1 << 24), "bns_spmm_sum_f32: bad feature width %lld", (long long)F);
    if (g->n_rows == 0) return BNS_OK;      // nothing to write (Y may legitimately be NULL)
    BNS_REQUIRE(Y, "bns_spmm_sum_f32: NULL output matrix");
    BNS_REQUIRE(X || g->nnz == 0, "bns_spmm_sum_f32: NULL input matrix");
    BNS_REQUIRE(ldx >= F && ldy >= F, "bns_spmm_sum_f32: leading dimension smaller than F");
    const size_t need = bns_spmm_workspace_bytes(g, F);
    if (need > 0 && (ws == nullptr || ws_bytes < need))
        return fail(BNS_E_WORKSPACE, "bns_spmm_sum_f32: workspace %zu bytes < %zu needed", ws_bytes, need);
    if (col_map == nullptr) n_direct = g->n_cols;
    BNS_REQUIRE(n_direct >= 0 && n_direct <= g->n_cols, "bns_spmm_sum_f32: n_direct out of range");
    if (x_rows <= 0) x_rows = g->n_cols;
    SpmmArgs a;
    a.indptr = g->indptr; a.indices = g->indices;
    a.chunk_row = g->chunk_row; a.chunk_start = g->chunk_start; a.chunk_part = g->chunk_part; a.chunk_cnt = nullptr;
    a.split_row = g->split_row; a.split_part = g->split_part;
    a.n_chunks = g->n_chunks; a.n_split = g->n_split; a.chunk_nnz = g->chunk_nnz;
    a.X = X; a.ldx = ldx; a.Y = Y; a.ldy = ldy; a.F = (int32_t)F;
    a.row_scale = row_scale; a.col_scale = col_scale; a.edge_weight = edge_weight; a.row_map = row_map; a.col_map = col_map;
    a.edge_perm = nullptr; a.edge_ld = 1;
    a.n_direct = (int32_t)n_direct; a.accumulate = accumulate ? 1 : 0;
    a.ws = reinterpret_cast<float *>(ws); a.ldws = ws_ld(F);
    a.n_tiles = 1;
    return spmm_dispatch(a, x_rows, slab_hint, as_stream(stream));
}

// The same kernel over the per-epoch compacted indices of bns_graph_compact_cols: `cidx` already holds rows of X, the
// chunk's live entries come first in its range, `chunk_cnt` says how many; `cw` = per-entry weights gathered at
// compaction time (GCN's 1/sqrt(out_deg) of the halo sources) or NULL.  Work is proportional to the SAMPLE, not to the
// halo (VERDICT r1 weak #3: the col_map kernel walks every halo edge to use ~10 % of them).
extern "C" int bns_spmm_compact_f32(const bns_graph_t *g, const int32_t *cidx, const float *cw, int64_t cw_ld,
                                    const int32_t *chunk_cnt, const float *X, int64_t ldx, int64_t F, float *Y, int64_t ldy,
                                    const float *row_scale, int64_t x_rows, int32_t slab_hint, int accumulate, void *ws,
                                    size_t ws_bytes, void *stream) {
    BNS_REQUIRE(g && cidx && chunk_cnt, "bns_spmm_compact_f32: NULL argument");
    BNS_REQUIRE(F > 0 && F < (1 << 24), "bns_spmm_compact_f32: bad feature width %lld", (long long)F);
    if (g->n_rows == 0) return BNS_OK;
    BNS_REQUIRE(Y && (X || g->nnz == 0), "bns_spmm_compact_f32: NULL matrix");
    BNS_REQUIRE(ldx >= F && ldy >= F, "bns_spmm_compact_f32: leading dimension smaller than F");
    const size_t need = bns_spmm_workspace_bytes(g, F);
    if (need > 0 && (ws == nullptr || ws_bytes < need))
        return fail(BNS_E_WORKSPACE, "bns_spmm_compact_f32: workspace %zu bytes < %zu needed", ws_bytes, need);
    SpmmArgs a;
    a.indptr = g->indptr; a.indices = cidx;
    a.chunk_row = g->chunk_row; a.chunk_start = g->chunk_start; a.chunk_part = g->chunk_part; a.chunk_cnt = chunk_cnt;
    a.split_row = g->split_row; a.split_part = g->split_part;
    a.n_chunks = g->n_chunks; a.n_split = g->n_split; a.chunk_nnz = g->chunk_nnz;
    a.X = X; a.ldx = ldx; a.Y = Y; a.ldy = ldy; a.F = (int32_t)F;
    a.row_scale = row_scale; a.col_scale = nullptr; a.edge_weight = cw; a.row_map = nullptr; a.col_map = nullptr;
    a.edge_perm = nullptr; a.edge_ld = cw_ld > 0 ? cw_ld : 1;
    a.n_direct = (int32_t)g->n_cols; a.accumulate = accumulate ? 1 : 0;
    a.ws = reinterpret_cast<float *>(ws); a.ldws = ws_ld(F);
    a.n_tiles = 1;
    return spmm_dispatch(a, x_rows > 0 ? x_rows : g->n_cols, slab_hint, as_stream(stream));
}

// Y[orow(r)] (+)= sum_k w_k X[c_k] with w_k = weights[(perm ? perm[k] : k) * ldw]: the weighted aggregation of GATConv
// (u_mul_e + sum) and -- on a transpose, with perm = its entry permutation (perm_from_transpose != 0) -- its gradient with
// respect to the source features, the attention staying in the order of the forward graph ([nnz, heads], one head per call).
extern "C" int bns_spmm_weighted_f32(const bns_graph_t *g, const float *X, int64_t ldx, int64_t F, float *Y, int64_t ldy,
                                     const float *weights, int64_t ldw, int perm_from_transpose, const int32_t *row_map,
                                     int64_t x_rows, int accumulate, void *ws, size_t ws_bytes, void *stream) {
    BNS_REQUIRE(g && weights, "bns_spmm_weighted_f32: NULL argument");
    BNS_REQUIRE(F > 0 && F < (1 << 24) && ldw >= 1, "bns_spmm_weighted_f32: bad width");
    BNS_REQUIRE(!perm_from_transpose || g->perm, "bns_spmm_weighted_f32: not a graph made by bns_graph_transpose");
    if (g->n_rows == 0) return BNS_OK;
    BNS_REQUIRE(Y && (X || g->nnz == 0) && ldx >= F && ldy >= F, "bns_spmm_weighted_f32: bad matrix");
    const size_t need = bns_spmm_workspace_bytes(g, F);
    if (need > 0 && (ws == nullptr || ws_bytes < need))
        return fail(BNS_E_WORKSPACE, "bns_spmm_weighted_f32: workspace %zu bytes < %zu needed", ws_bytes, need);
    SpmmArgs a;
    a.indptr = g->indptr; a.indices = g->indices;
    a.chunk_row = g->chunk_row; a.chunk_start = g->chunk_start; a.chunk_part = g->chunk_part; a.chunk_cnt = nullptr;
    a.split_row = g->split_row; a.split_part = g->split_part;
    a.n_chunks = g->n_chunks; a.n_split = g->n_split; a.chunk_nnz = g->chunk_nnz;
    a.X = X; a.ldx = ldx; a.Y = Y; a.ldy = ldy; a.F = (int32_t)F;
    a.row_scale = nullptr; a.col_scale = nullptr; a.edge_weight = weights; a.row_map = row_map; a.col_map = nullptr;
    a.edge_perm = perm_from_transpose ? g->perm : nullptr; a.edge_ld = ldw;
    a.n_direct = (int32_t)g->n_cols; a.accumulate = accumulate ? 1 : 0;
    a.ws = reinterpret_cast<float *>(ws); a.ldws = ws_ld(F);
    a.n_tiles = 1;
    return spmm_dispatch(a, x_rows > 0 ? x_rows : g->n_cols, 0, as_stream(stream));
}

// =================================================================================================
// SDDMM (dot): out[k] = < A[arow(r), :], B[xrow(c_k), :] > for every entry k of row r
// (the attention gradient of GAT: d a_uv = <dOut[v], ft[u]>, the transpose partner of the weighted SpMM)
// =================================================================================================
namespace {

struct SddmmArgs {
    const int64_t *indptr;
    const int32_t *indices;
    const int32_t *chunk_row;
    const int64_t *chunk_start;
    int64_t n_chunks;
    int32_t chunk_nnz;
    const float *A; int64_t lda;
    const float *B; int64_t ldb;
    int32_t F;
    const int32_t *row_map, *col_map;
    int32_t n_direct;
    float *out; int64_t ldo;          // out[k * ldo]
};

// one warp per chunk; the lanes keep their slice of A[row] in registers and walk the entries like the SpMM does
template <int NV, int U>
__global__ void __launch_bounds__(kThreads) sddmm_dot_kernel(SddmmArgs a) {
    __shared__ int32_t s_col[kWarps][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t warps_total = (int64_t)gridDim.x * kWarps;
    for (int64_t c = (int64_t)blockIdx.x * kWarps + w; c < a.n_chunks; c += warps_total) {
        const int32_t row = a.chunk_row[c];
        const int64_t s = a.chunk_start[c];
        int64_t e = a.indptr[row + 1];
        if (e > s + a.chunk_nnz) e = s + a.chunk_nnz;
        int32_t arow = row;
        if (a.row_map) arow = a.row_map[row];
        float4 av[NV];
#pragma unroll
        for (int t = 0; t < NV; ++t) {
            const int f = (lane + 32 * t) * 4;
            av[t] = (arow >= 0 && f < a.F) ? *reinterpret_cast<const float4 *>(a.A + (int64_t)arow * a.lda + f)
                                            : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        for (int64_t k0 = s; k0 < e; k0 += 32) {
            const int64_t k = k0 + lane;
            int32_t col = -1;
            if (k < e) {
                col = ld_stream_i32(a.indices + k);
                if (a.col_map && col >= a.n_direct) col = __ldg(a.col_map + (col - a.n_direct));
                if (arow < 0) col = -1;
            }
            s_col[w][lane] = col;
            __syncwarp();
            const int cnt = (e - k0) < 32 ? (int)(e - k0) : 32;
            float mine = 0.f;
            // U gathered rows in flight per lane (the loads of one group are issued before any of its sums)
            for (int j0 = 0; j0 < cnt; j0 += U) {
                float4 b[U][NV];
                int32_t cj[U];
#pragma unroll
                for (int q = 0; q < U; ++q) {
                    cj[q] = (j0 + q < cnt) ? s_col[w][j0 + q] : -1;
#pragma unroll
                    for (int t = 0; t < NV; ++t) {
                        const int f = (lane + 32 * t) * 4;
                        b[q][t] = (cj[q] >= 0 && f < a.F)
                                      ? __ldg(reinterpret_cast<const float4 *>(a.B + (int64_t)cj[q] * a.ldb + f))
                                      : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                }
                float d[U];
#pragma unroll
                for (int q = 0; q < U; ++q) {
                    d[q] = 0.f;
#pragma unroll
                    for (int t = 0; t < NV; ++t)
                        d[q] += (av[t].x * b[q][t].x + av[t].y * b[q][t].y) + (av[t].z * b[q][t].z + av[t].w * b[q][t].w);
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
                    for (int q = 0; q < U; ++q) d[q] += __shfl_xor_sync(0xffffffffu, d[q], o);
                }
#pragma unroll
                for (int q = 0; q < U; ++q)
                    if (lane == j0 + q) mine = d[q];
            }
            if (k < e) a.out[k * a.ldo] = mine;
            __syncwarp();
        }
    }
}

}  // namespace

extern "C" int bns_sddmm_dot_f32(const bns_graph_t *g, const float *A, int64_t lda, const float *B, int64_t ldb, int64_t F,
                                 const int32_t *row_map, const int32_t *col_map, int64_t n_direct, float *out,
                                 int64_t ldo, void *stream) {
    BNS_REQUIRE(g, "bns_sddmm_dot_f32: NULL graph");
    BNS_REQUIRE(F > 0 && F % 4 == 0 && F <= 1024, "bns_sddmm_dot_f32: need F %% 4 == 0 and F <= 1024 (got %lld)", (long long)F);
    if (g->nnz == 0) return BNS_OK;
    BNS_REQUIRE(A && B && out, "bns_sddmm_dot_f32: NULL pointer");
    BNS_REQUIRE(lda % 4 == 0 && ldb % 4 == 0 && lda >= F && ldb >= F && ldo >= 1, "bns_sddmm_dot_f32: bad leading dimension");
    BNS_REQUIRE(((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(B)) % 16) == 0, "bns_sddmm_dot_f32: unaligned");
    if (col_map == nullptr) n_direct = g->n_cols;
    SddmmArgs a;
    a.indptr = g->indptr; a.indices = g->indices; a.chunk_row = g->chunk_row; a.chunk_start = g->chunk_start;
    a.n_chunks = g->n_chunks; a.chunk_nnz = g->chunk_nnz;
    a.A = A; a.lda = lda; a.B = B; a.ldb = ldb; a.F = (int32_t)F; a.row_map = row_map; a.col_map = col_map;
    a.n_direct = (int32_t)n_direct; a.out = out; a.ldo = ldo;
    int64_t want = (a.n_chunks + kWarps - 1) / kWarps, cap = (int64_t)sm_count() * 6;
    unsigned gx = (unsigned)(want < cap ? (want > 0 ? want : 1) : cap);
    cudaStream_t st = as_stream(stream);
    const int nv = (int)((F + 127) / 128);
    // gathered rows in flight per lane, measured on the Yelp shape (profiles/gat_r02.md): F = 256: 8 (3.2 ms) beats 4 (3.9 ms);
    // F = 100: 4 (1.46 ms) beats 8 (1.76 ms)
    if (nv <= 1) sddmm_dot_kernel<1, 4><<<gx, kThreads, 0, st>>>(a);
    else if (nv == 2) sddmm_dot_kernel<2, 8><<<gx, kThreads, 0, st>>>(a);
    else if (nv <= 4) sddmm_dot_kernel<4, 2><<<gx, kThreads, 0, st>>>(a);
    else sddmm_dot_kernel<8, 1><<<gx, kThreads, 0, st>>>(a);
    ++g_launches;
    BNS_CUDA(cudaGetLastError());
    return BNS_OK;
}

// =================================================================================================
// boundary pack / scatter / copy
// =================================================================================================
namespace {

// one warp per row, 16-byte lanes when aligned
template <bool VEC, bool SCATTER>
__global__ void __launch_bounds__(kThreads) rows_kernel(const float *__restrict__ src, int64_t lds, float *dst,
                                                        int64_t ldd, const int64_t *__restrict__ idx, int64_t k,
                                                        int32_t F, float div) {
    const int lane = threadIdx.x & 31;
    const int64_t warps_total = (int64_t)gridDim.x * kWarps;
    for (int64_t i = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); i < k; i += warps_total) {
        const int64_t r = idx ? idx[i] : i;
        const float *s = SCATTER ? src + i * lds : src + r * lds;
        float *d = SCATTER ? dst + r * ldd : dst + i * ldd;
        if (VEC) {
            for (int f = lane * 4; f < F; f += 128) {
                float4 v = *reinterpret_cast<const float4 *>(s + f);
                v.x = __fdiv_rn(v.x, div); v.y = __fdiv_rn(v.y, div); v.z = __fdiv_rn(v.z, div); v.w = __fdiv_rn(v.w, div);
                if (SCATTER) {
                    float4 o = *reinterpret_cast<float4 *>(d + f);
                    v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
                }
                *reinterpret_cast<float4 *>(d + f) = v;
            }
        } else {
            for (int f = lane; f < F; f += 32) {
                float v = __fdiv_rn(s[f], div);
                if (SCATTER) v += d[f];
                d[f] = v;
            }
        }
    }
}

inline bool vec_ok(const void *a, const void *b, int64_t F, int64_t lda, int64_t ldb) {
    return F % 4 == 0 && lda % 4 == 0 && ldb % 4 == 0 &&
           ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) % 16 == 0);
}

inline unsigned rows_grid(int64_t k) {
    int64_t want = (k + kWarps - 1) / kWarps;
    int64_t cap = (int64_t)sm_count() * 8;
    return (unsigned)(want < cap ? (want > 0 ? want : 1) : cap);
}

}  // namespace

extern "C" int bns_gather_div_f32(const float *H, int64_t ldh, int64_t F, const int64_t *idx, int64_t k, float div,
                                  float *out, int64_t ldo, void *stream) {
    BNS_REQUIRE(k >= 0 && F > 0, "bns_gather_div_f32: bad size");
    if (k == 0) return BNS_OK;
    BNS_REQUIRE(H && out && idx, "bns_gather_div_f32: NULL pointer");
    BNS_REQUIRE(ldh >= F && ldo >= F, "bns_gather_div_f32: leading dimension smaller than F");
    BNS_REQUIRE(div != 0.f, "bns_gather_div_f32: division by zero");
    cudaStream_t st = as_stream(stream);
    if (vec_ok(H, out, F, ldh, ldo))
        rows_kernel<true, false><<<rows_grid(k), kThreads, 0, st>>>(H, ldh, out, ldo, idx, k, (int32_t)F, div);
    else
        rows_kernel<false, false><<<rows_grid(k), kThreads, 0, st>>>(H, ldh, out, ldo, idx, k, (int32_t)F, div);
    ++g_launches;
    BNS_CUDA(cudaGetLastError());
    return BNS_OK;
}

extern "C" int bns_scatter_add_div_f32(float *G, int64_t ldg, int64_t F, const int64_t *idx, int64_t k, float div,
                                       const float *src, int64_t lds, void *stream) {
    BNS_REQUIRE(k >= 0 && F > 0, "bns_scatter_add_div_f32: bad size");
    if (k == 0) return BNS_OK;
    BNS_REQUIRE(G && src && idx, "bns_scatter_add_div_f32: NULL pointer");
    BNS_REQUIRE(ldg >= F && lds >= F, "bns_scatter_add_div_f32: leading dimension smaller than F");
    BNS_REQUIRE(div != 0.f, "bns_scatter_add_div_f32: division by zero");
    cudaStream_t st = as_stream(stream);
    if (vec_ok(G, src, F, ldg, lds))
        rows_kernel<true, true><<<rows_grid(k), kThreads, 0, st>>>(src, lds, G, ldg, idx, k, (int32_t)F, div);
    else
        rows_kernel<false, true><<<rows_grid(k), kThreads, 0, st>>>(src, lds, G, ldg, idx, k, (int32_t)F, div);
    ++g_launches;
    BNS_CUDA(cudaGetLastError());
    return BNS_OK;
}

extern "C" int bns_copy_rows_f32(const float *src, int64_t lds, float *dst, int64_t ldd, int64_t n_rows, int64_t F,
                                 void *stream) {
    BNS_REQUIRE(n_rows >= 0 && F > 0, "bns_copy_rows_f32: bad size");
    if (n_rows == 0) return BNS_OK;
    BNS_REQUIRE(src && dst, "bns_copy_rows_f32: NULL pointer");
    BNS_REQUIRE(lds >= F && ldd >= F, "bns_copy_rows_f32: leading dimension smaller than F");
    BNS_CUDA(cudaMemcpy2DAsync(dst, ldd * sizeof(float), src, lds * sizeof(float), F * sizeof(float), n_rows,
                               cudaMemcpyDeviceToDevice, as_stream(stream)));
    return BNS_OK;
}

// =================================================================================================
// sampler
// =================================================================================================
namespace {

__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t out[4]) {
    constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0;
        const uint32_t hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += W0; k1 += W1;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__global__ void sample_keys_kernel(const int64_t *__restrict__ seg_begin, int32_t n_seg, int64_t B, uint64_t seed,
                                   uint64_t offset, const uint64_t *__restrict__ offset_dev,
                                   uint64_t *__restrict__ keys, int32_t *__restrict__ vals) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= B) return;
    if (offset_dev) offset += *offset_dev;      // CUDA-graph replays: the epoch counter lives on the device
    int32_t lo = 0, hi = n_seg;   // segment s with seg_begin[s] <= i < seg_begin[s+1]
    while (hi - lo > 1) {
        const int32_t mid = (lo + hi) >> 1;
        if (seg_begin[mid] <= i) lo = mid; else hi = mid;
    }
    uint32_t r[4];
    philox4x32_10((uint32_t)i, (uint32_t)((uint64_t)i >> 32), (uint32_t)offset, (uint32_t)(offset >> 32),
                  (uint32_t)seed, (uint32_t)(seed >> 32), r);
    const uint64_t r56 = ((uint64_t)r[0] << 24) | (uint64_t)(r[1] >> 8);
    keys[i] = ((uint64_t)lo << 56) | r56;
    vals[i] = (int32_t)i;
}

__global__ void sample_take_kernel(const int64_t *__restrict__ boundary_cat, const int64_t *__restrict__ seg_begin,
                                   const int64_t *__restrict__ out_begin, int32_t n_seg, int64_t K,
                                   const int32_t *__restrict__ sorted_vals, int64_t *__restrict__ selected) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= K) return;
    int32_t lo = 0, hi = n_seg;
    while (hi - lo > 1) {
        const int32_t mid = (lo + hi) >> 1;
        if (out_begin[mid] <= t) lo = mid; else hi = mid;
    }
    const int64_t j = t - out_begin[lo];
    selected[t] = boundary_cat[sorted_vals[seg_begin[lo] + j]];
}

struct SampleLayout {
    size_t keys_in, keys_out, vals_in, vals_out, tmp, tmp_bytes, total;
};

inline size_t align256(size_t x) { return (x + 255) / 256 * 256; }

SampleLayout sample_layout(int64_t B) {
    SampleLayout l;
    size_t n = (size_t)(B > 0 ? B : 1);
    l.keys_in = 0;
    l.keys_out = l.keys_in + align256(n * 8);
    l.vals_in = l.keys_out + align256(n * 8);
    l.vals_out = l.vals_in + align256(n * 4);
    l.tmp = l.vals_out + align256(n * 4);
    size_t tb = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tb, (const uint64_t *)nullptr, (uint64_t *)nullptr,
                                    (const int32_t *)nullptr, (int32_t *)nullptr, (int)n, 0, 64, (cudaStream_t)0);
    l.tmp_bytes = align256(tb ? tb : 16);
    l.total = l.tmp + l.tmp_bytes;
    return l;
}

}  // namespace

extern "C" size_t bns_sample_workspace_bytes(int64_t B) { return sample_layout(B).total; }

extern "C" int bns_sample_boundary(const int64_t *boundary_cat, const int64_t *seg_begin, const int64_t *out_begin,
                                   int32_t n_seg, int64_t B, int64_t K_total, uint64_t seed, uint64_t offset,
                                   const uint64_t *offset_dev,
                                   int64_t *selected, void *ws, size_t ws_bytes, void *stream) {
    BNS_REQUIRE(n_seg >= 0 && n_seg <= 255, "bns_sample_boundary: n_seg must be in [0, 255]");
    BNS_REQUIRE(B >= 0 && K_total >= 0 && K_total <= B, "bns_sample_boundary: need 0 <= K_total <= B");
    BNS_REQUIRE(B < INT32_MAX, "bns_sample_boundary: B >= 2^31");
    if (K_total == 0 || n_seg == 0) return BNS_OK;
    BNS_REQUIRE(boundary_cat && seg_begin && out_begin && selected, "bns_sample_boundary: NULL pointer");
    const SampleLayout l = sample_layout(B);
    if (!ws || ws_bytes < l.total)
        return fail(BNS_E_WORKSPACE, "bns_sample_boundary: workspace %zu bytes < %zu needed", ws_bytes, l.total);
    char *base = reinterpret_cast<char *>(ws);
    uint64_t *keys_in = reinterpret_cast<uint64_t *>(base + l.keys_in);
    uint64_t *keys_out = reinterpret_cast<uint64_t *>(base + l.keys_out);
    int32_t *vals_in = reinterpret_cast<int32_t *>(base + l.vals_in);
    int32_t *vals_out = reinterpret_cast<int32_t *>(base + l.vals_out);
    cudaStream_t st = as_stream(stream);
    sample_keys_kernel<<<(unsigned)((B + 255) / 256), 256, 0, st>>>(seg_begin, n_seg, B, seed, offset, offset_dev, keys_in, vals_in);
    size_t tb = l.tmp_bytes;
    BNS_CUDA(cub::DeviceRadixSort::SortPairs(base + l.tmp, tb, keys_in, keys_out, vals_in, vals_out, (int)B, 0, 64, st));
    sample_take_kernel<<<(unsigned)((K_total + 255) / 256), 256, 0, st>>>(boundary_cat, seg_begin, out_begin, n_seg,
                                                                         K_total, vals_out, selected);
    g_launches += 2;
    BNS_CUDA(cudaGetLastError());
    return BNS_OK;
}

// =================================================================================================
// fused LayerNorm -> ReLU -> dropout  (module/model.py:88-91 then :45/:80 of the next layer)
// =================================================================================================
namespace {

constexpr int kLnMaxNV = 8;      // F <= 1024

struct LnArgs {
    const float *x; int64_t ldx;
    const float *dy; int64_t lddy;
    float *y; int64_t ldy;          // forward output / backward dx
    const float *gamma, *beta;
    float *mean, *rstd;
    int64_t n; int32_t F;
    float eps, p, keep_scale;
    uint64_t seed, offset;
    const uint64_t *offset_dev;
    float *partial;                 // backward: [gridDim.x][2][F] column partial sums (dgamma, dbeta)
};

// keep-mask of the 4 elements of vector `vec` of row `row`: one Philox4x32-10 call
__device__ __forceinline__ void drop_mask4(uint64_t seed, uint64_t offset, int64_t row, int vec, float p, bool keep[4]) {
    uint32_t r[4];
    philox4x32_10((uint32_t)row, (uint32_t)((uint64_t)row >> 32) ^ ((uint32_t)vec << 8), (uint32_t)offset,
                  (uint32_t)(offset >> 32), (uint32_t)seed, (uint32_t)(seed >> 32), r);
#pragma unroll
    for (int i = 0; i < 4; ++i) keep[i] = (float)r[i] * 2.3283064365386963e-10f >= p;
}

template <int NV, bool BACKWARD>
__global__ void __launch_bounds__(kThreads) ln_relu_dropout_kernel(LnArgs a) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t warps_total = (int64_t)gridDim.x * kWarps;
    const uint64_t offset = a.offset + (a.offset_dev ? *a.offset_dev : 0ull);
    const float invF = 1.f / (float)a.F;
    float4 g4[NV], b4[NV];
    float4 sg[NV], sb[NV];             // backward: this warp's column sums of dgamma / dbeta
    bool ok[NV];
#pragma unroll
    for (int t = 0; t < NV; ++t) {
        const int f = (lane + 32 * t) * 4;
        ok[t] = f < a.F;
        g4[t] = ok[t] ? *reinterpret_cast<const float4 *>(a.gamma + f) : make_float4(0.f, 0.f, 0.f, 0.f);
        b4[t] = ok[t] ? *reinterpret_cast<const float4 *>(a.beta + f) : make_float4(0.f, 0.f, 0.f, 0.f);
        sg[t] = make_float4(0.f, 0.f, 0.f, 0.f);
        sb[t] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    for (int64_t row = (int64_t)blockIdx.x * kWarps + w; row < a.n; row += warps_total) {
        float4 v[NV];
        float s = 0.f;
#pragma unroll
        for (int t = 0; t < NV; ++t) {
            v[t] = ok[t] ? *reinterpret_cast<const float4 *>(a.x + row * a.ldx + (lane + 32 * t) * 4)
                         : make_float4(0.f, 0.f, 0.f, 0.f);
            s += (v[t].x + v[t].y) + (v[t].z + v[t].w);
        }
        float mean, rstd;
        if (!BACKWARD) {
            mean = warp_sum(s) * invF;
            float q = 0.f;
#pragma unroll
            for (int t = 0; t < NV; ++t) {
                if (!ok[t]) continue;
                const float dx = v[t].x - mean, dy = v[t].y - mean, dz = v[t].z - mean, dw = v[t].w - mean;
                q += (dx * dx + dy * dy) + (dz * dz + dw * dw);
            }
            rstd = rsqrtf(warp_sum(q) * invF + a.eps);
            if (lane == 0) { a.mean[row] = mean; a.rstd[row] = rstd; }
        } else {
            mean = a.mean[row];
            rstd = a.rstd[row];
        }
        float4 gz[NV];                 // backward: dL/dz * gamma ; forward: unused
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int t = 0; t < NV; ++t) {
            if (!ok[t]) continue;
            const int f = (lane + 32 * t) * 4;
            bool keep[4] = {true, true, true, true};
            if (a.p > 0.f) drop_mask4(a.seed, offset, row, lane + 32 * t, a.p, keep);
            float xh[4] = {(v[t].x - mean) * rstd, (v[t].y - mean) * rstd, (v[t].z - mean) * rstd, (v[t].w - mean) * rstd};
            const float gg[4] = {g4[t].x, g4[t].y, g4[t].z, g4[t].w}, bb[4] = {b4[t].x, b4[t].y, b4[t].z, b4[t].w};
            if (!BACKWARD) {
                float o[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float z = fmaf(xh[i], gg[i], bb[i]);
                    o[i] = (z > 0.f && keep[i]) ? z * a.keep_scale : 0.f;
                }
                *reinterpret_cast<float4 *>(a.y + row * a.ldy + f) = make_float4(o[0], o[1], o[2], o[3]);
            } else {
                const float4 d4 = *reinterpret_cast<const float4 *>(a.dy + row * a.lddy + f);
                const float dd[4] = {d4.x, d4.y, d4.z, d4.w};
                float gzz[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float z = fmaf(xh[i], gg[i], bb[i]);
                    const float g = (z > 0.f && keep[i]) ? dd[i] * a.keep_scale : 0.f;      // dL/dz
                    (&sg[t].x)[i] += g * xh[i];
                    (&sb[t].x)[i] += g;
                    gzz[i] = g * gg[i];                                                     // dL/dxhat
                    s1 += gzz[i];
                    s2 += gzz[i] * xh[i];
                }
                gz[t] = make_float4(gzz[0], gzz[1], gzz[2], gzz[3]);
                v[t] = make_float4(xh[0], xh[1], xh[2], xh[3]);
            }
        }
        if (BACKWARD) {
            s1 = warp_sum(s1) * invF;
            s2 = warp_sum(s2) * invF;
#pragma unroll
            for (int t = 0; t < NV; ++t) {
                if (!ok[t]) continue;
                const int f = (lane + 32 * t) * 4;
                float4 o;
                o.x = rstd * (gz[t].x - s1 - v[t].x * s2);
                o.y = rstd * (gz[t].y - s1 - v[t].y * s2);
                o.z = rstd * (gz[t].z - s1 - v[t].z * s2);
                o.w = rstd * (gz[t].w - s1 - v[t].w * s2);
                *reinterpret_cast<float4 *>(a.y + row * a.ldy + f) = o;
            }
        }
    }
    if (BACKWARD) {      // CTA-level column sums, warps added in a fixed order -> one partial row per CTA
        __shared__ float red[2][NV * 128];
        for (int i = threadIdx.x; i < 2 * NV * 128; i += kThreads) (&red[0][0])[i] = 0.f;
        __syncthreads();
        for (int ww = 0; ww < kWarps; ++ww) {
            if (w == ww) {
#pragma unroll
                for (int t = 0; t < NV; ++t) {
                    const int f = (lane + 32 * t) * 4;
                    if (!ok[t]) continue;
                    float4 r0 = *reinterpret_cast<float4 *>(&red[0][f]), r1 = *reinterpret_cast<float4 *>(&red[1][f]);
                    r0.x += sg[t].x; r0.y += sg[t].y; r0.z += sg[t].z; r0.w += sg[t].w;
                    r1.x += sb[t].x; r1.y += sb[t].y; r1.z += sb[t].z; r1.w += sb[t].w;
                    *reinterpret_cast<float4 *>(&red[0][f]) = r0;
                    *reinterpret_cast<float4 *>(&red[1][f]) = r1;
                }
            }
            __syncthreads();
        }
        for (int i = threadIdx.x; i < 2 * a.F; i += kThreads) {
            const int which = i / a.F, f = i % a.F;
            a.partial[((int64_t)blockIdx.x * 2 + which) * a.F + f] = red[which][f];
        }
    }
}

// one warp per output column (2F of them: dgamma then dbeta): lanes stride over the per-CTA partials, fixed shuffle tree
__global__ void __launch_bounds__(kThreads) ln_colsum_kernel(const float *__restrict__ partial, int n_part, int F,
                                                             float *__restrict__ dgamma, float *__restrict__ dbeta) {
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * kWarps + (threadIdx.x >> 5);
    if (i >= 2 * F) return;
    const int which = i / F, f = i % F;
    float acc = 0.f;
    for (int p = lane; p < n_part; p += 32) acc += partial[((int64_t)p * 2 + which) * F + f];
    acc = warp_sum(acc);
    if (lane == 0) (which == 0 ? dgamma : dbeta)[f] = acc;
}

inline unsigned ln_grid(int64_t n) {
    int64_t want = (n + kWarps - 1) / kWarps;
    int64_t cap = (int64_t)sm_count() * 4;
    return (unsigned)(want < cap ? (want > 0 ? want : 1) : cap);
}

template <bool BWD>
int launch_ln(const LnArgs &a, unsigned grid, cudaStream_t st) {
    const int nv = (a.F + 127) / 128;
    switch (nv) {
        case 1: ln_relu_dropout_kernel<1, BWD><<<grid, kThreads, 0, st>>>(a); break;
        case 2: ln_relu_dropout_kernel<2, BWD><<<grid, kThreads, 0, st>>>(a); break;
        case 3: case 4: ln_relu_dropout_kernel<4, BWD><<<grid, kThreads, 0, st>>>(a); break;
        default: ln_relu_dropout_kernel<8, BWD><<<grid, kThreads, 0, st>>>(a); break;
    }
    return BNS_OK;
}

}  // namespace

extern "C" size_t bns_ln_bwd_workspace_bytes(int64_t F) { return (size_t)sm_count() * 4 * 2 * (size_t)F * sizeof(float); }

extern "C" int bns_ln_relu_dropout_fwd_f32(const float *x, int64_t ldx, int64_t n, int64_t F, const float *gamma,
                                           const float *beta, float eps, float p, uint64_t seed, uint64_t offset,
                                           const uint64_t *offset_dev, float *y, int64_t ldy, float *mean, float *rstd,
                                           void *stream) {
    BNS_REQUIRE(n >= 0 && F > 0 && F % 4 == 0 && F <= kLnMaxNV * 128, "bns_ln_relu_dropout_fwd_f32: need F %% 4 == 0, F <= 1024");
    if (n == 0) return BNS_OK;
    BNS_REQUIRE(x && y && gamma && beta && mean && rstd, "bns_ln_relu_dropout_fwd_f32: NULL pointer");
    BNS_REQUIRE(ldx % 4 == 0 && ldy % 4 == 0 && ldx >= F && ldy >= F, "bns_ln_relu_dropout_fwd_f32: bad leading dimension");
    BNS_REQUIRE(p >= 0.f && p < 1.f, "bns_ln_relu_dropout_fwd_f32: p must be in [0, 1)");
    LnArgs a{};
    a.x = x; a.ldx = ldx; a.y = y; a.ldy = ldy; a.gamma = gamma; a.beta = beta; a.mean = mean; a.rstd = rstd;
    a.n = n; a.F = (int32_t)F; a.eps = eps; a.p = p; a.keep_scale = 1.f / (1.f - p);
    a.seed = seed; a.offset = offset; a.offset_dev = offset_dev;
    launch_ln<false>(a, ln_grid(n), as_stream(stream));
    ++g_launches;
    BNS_CUDA(cudaGetLastError());
    return BNS_OK;
}

extern "C" int bns_ln_relu_dropout_bwd_f32(const float *dy, int64_t lddy, const float *x, int64_t ldx, int64_t n, int64_t F,
                                           const float *gamma, const float *beta, const float *mean, const float *rstd,
                                           float eps, float p, uint64_t seed, uint64_t offset, const uint64_t *offset_dev,
                                           float *dx, int64_t lddx, float *dgamma, float *dbeta, void *ws, size_t ws_bytes,
                                           void *stream) {
    BNS_REQUIRE(n >= 0 && F > 0 && F % 4 == 0 && F <= kLnMaxNV * 128, "bns_ln_relu_dropout_bwd_f32: need F %% 4 == 0, F <= 1024");
    BNS_REQUIRE(dy && x && dx && gamma && beta && mean && rstd && dgamma && dbeta, "bns_ln_relu_dropout_bwd_f32: NULL pointer");
    BNS_REQUIRE(ldx % 4 == 0 && lddy % 4 == 0 && lddx % 4 == 0, "bns_ln_relu_dropout_bwd_f32: bad leading dimension");
    const unsigned grid = ln_grid(n > 0 ? n : 1);
    if (!ws || ws_bytes < (size_t)grid * 2 * F * sizeof(float))
        return fail(BNS_E_WORKSPACE, "bns_ln_relu_dropout_bwd_f32: workspace too small");
    LnArgs a{};
    a.x = x; a.ldx = ldx; a.dy = dy; a.lddy = lddy; a.y = dx; a.ldy = lddx; a.gamma = gamma; a.beta = beta;
    a.mean = const_cast<float *>(mean); a.rstd = const_cast<float *>(rstd);
    a.n = n; a.F = (int32_t)F; a.eps = eps; a.p = p; a.keep_scale = 1.f / (1.f - p);
    a.seed = seed; a.offset = offset; a.offset_dev = offset_dev; a.partial = reinterpret_cast<float *>(ws);
    cudaStream_t st = as_stream(stream);
    launch_ln<true>(a, grid, st);
    ln_colsum_kernel<<<(unsigned)((2 * F + kWarps - 1) / kWarps), kThreads, 0, st>>>(a.partial, (int)grid, (int)F, dgamma, dbeta);
    g_launches += 2;
    BNS_CUDA(cudaGetLastError());
    return BNS_OK;
}

// =================================================================================================
// column sums (bias gradients of the dense layers: db = dY.sum(0)), deterministic two-pass
// =================================================================================================
namespace {

constexpr int kColsumMaxCols = 1024;

// block b sums rows b, b + gridDim.x, ... ; thread (rg, c) = (t / CV, t % CV) owns float4 column c of every RG-th of them
__global__ void __launch_bounds__(kThreads) colsum_partial_kernel(const float *__restrict__ X, int64_t ld, int64_t rows, int CV,
                                                                 float4 *__restrict__ partial) {
    __shared__ float4 s_acc[kThreads];
    const int RG = kThreads / CV;
    const int rg = threadIdx.x / CV, c = threadIdx.x % CV;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (rg < RG) {
        // contiguous row range per block, rows interleaved over the row groups inside it
        const int64_t per = (rows + gridDim.x - 1) / gridDim.x;
        const int64_t r0 = (int64_t)blockIdx.x * per, r1 = r0 + per < rows ? r0 + per : rows;
        for (int64_t r = r0 + rg; r < r1; r += RG) {
            const float4 v = __ldg(reinterpret_cast<const float4 *>(X + r * ld) + c);
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
    }
    s_acc[threadIdx.x] = acc;
    __syncthreads();
    if (rg == 0) {
        for (int g = 1; g < RG; ++g) {
            const float4 v = s_acc[g * CV + c];
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
        partial[(int64_t)blockIdx.x * CV + c] = acc;
    }
}

// one warp per float4 column: lanes stride over the per-block partials, then a fixed shuffle tree (deterministic)
__global__ void __launch_bounds__(kThreads) colsum_final_kernel(const float4 *__restrict__ partial, int n_part, int CV,
                                                                float4 *__restrict__ out, float4 *__restrict__ out2) {
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * kWarps + (threadIdx.x >> 5);
    if (c >= CV) return;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int p = lane; p < n_part; p += 32) {
        const float4 v = partial[(int64_t)p * CV + c];
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    acc.x = warp_sum(acc.x); acc.y = warp_sum(acc.y); acc.z = warp_sum(acc.z); acc.w = warp_sum(acc.w);
    if (lane == 0) {
        out[c] = acc;
        if (out2) out2[c] = acc;
    }
}

inline int colsum_blocks() { return sm_count() * 4; }

}  // namespace

extern "C" size_t bns_colsum_workspace_bytes(int64_t cols) {
    return cols > 0 ? (size_t)colsum_blocks() * (size_t)((cols + 3) / 4) * sizeof(float4) : 0;
}

extern "C" int bns_colsum_f32(const float *X, int64_t ld, int64_t rows, int64_t cols, float *out, float *out2, void *ws,
                              size_t ws_bytes, void *stream) {
    BNS_REQUIRE(X && out, "bns_colsum_f32: NULL argument");
    BNS_REQUIRE(!out2 || (reinterpret_cast<uintptr_t>(out2) & 15u) == 0, "bns_colsum_f32: out2 must be 16-byte aligned");
    BNS_REQUIRE(rows > 0 && cols > 0 && cols % 4 == 0 && cols <= kColsumMaxCols, "bns_colsum_f32: need 0 < cols <= 1024, cols %% 4 == 0");
    BNS_REQUIRE(ld >= cols && ld % 4 == 0 && (reinterpret_cast<uintptr_t>(X) & 15u) == 0 && (reinterpret_cast<uintptr_t>(out) & 15u) == 0,
                "bns_colsum_f32: 16-byte aligned rows required");
    const size_t need = bns_colsum_workspace_bytes(cols);
    if (!ws || ws_bytes < need || (reinterpret_cast<uintptr_t>(ws) & 15u))
        return fail(BNS_E_WORKSPACE, "bns_colsum_f32: workspace %zu bytes < %zu needed", ws_bytes, need);
    const int CV = (int)(cols / 4);
    int blocks = colsum_blocks();
    if ((int64_t)blocks > rows) blocks = (int)rows;
    cudaStream_t st = as_stream(stream);
    colsum_partial_kernel<<<blocks, kThreads, 0, st>>>(X, ld, rows, CV, reinterpret_cast<float4 *>(ws));
    colsum_final_kernel<<<(CV + kWarps - 1) / kWarps, kThreads, 0, st>>>(reinterpret_cast<const float4 *>(ws), blocks, CV,
                                                                         reinterpret_cast<float4 *>(out),
                                                                         reinterpret_cast<float4 *>(out2));
    g_launches += 2;
    BNS_CUDA(cudaGetLastError());
    return BNS_OK;
}

// =================================================================================================
// halo slot map
// =================================================================================================
namespace {

__global__ void fill_i32_kernel(int32_t *dst, int64_t n, int32_t v) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) dst[i] = v;
}

__global__ void halo_slot_kernel(const int64_t *__restrict__ pos, const int64_t *__restrict__ one_hops, int64_t r,
                                 int64_t n_in, int32_t slab_offset, int32_t *__restrict__ slot) {
    int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= r) return;
    const int64_t local = pos[one_hops[k]];
    if (local >= n_in) slot[local - n_in] = slab_offset + (int32_t)k;
}

}  // namespace

extern "C" int bns_fill_i32(int32_t *dst, int64_t n, int32_t value, void *stream) {
    BNS_REQUIRE(n >= 0, "bns_fill_i32: negative size");
    if (n == 0) return BNS_OK;
    BNS_REQUIRE(dst, "bns_fill_i32: NULL pointer");
    fill_i32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, as_stream(stream)>>>(dst, n, value);
    ++g_launches;
    BNS_CUDA(cudaGetLastError());
    return BNS_OK;
}

extern "C" int bns_halo_slot_update(const int64_t *pos, const int64_t *one_hops, int64_t r, int64_t n_in,
                                    int32_t slab_offset, int32_t *slot, void *stream) {
    BNS_REQUIRE(r >= 0, "bns_halo_slot_update: negative size");
    if (r == 0) return BNS_OK;
    BNS_REQUIRE(pos && one_hops && slot, "bns_halo_slot_update: NULL pointer");
    halo_slot_kernel<<<(unsigned)((r + 255) / 256), 256, 0, as_stream(stream)>>>(pos, one_hops, r, n_in, slab_offset, slot);
    ++g_launches;
    BNS_CUDA(cudaGetLastError());
    return BNS_OK;
}

// =================================================================================================
// peer-mapped exchange
// =================================================================================================
struct bns_p2p {
    int32_t rank = 0, world = 0, n_flags = 0;
    size_t slab_bytes = 0;
    char *slab = nullptr;                 // this rank's receive slab
    unsigned long long *flags = nullptr;  // this rank's flag block
    char **peer_slab = nullptr;           // [world] mapped pointers (self = own)
    unsigned long long **peer_flags = nullptr;
    size_t *peer_slab_bytes = nullptr;    // [world] size of each peer's slab (bounds checks on puts)
    bool *imported = nullptr;             // opened with cudaIpcOpenMemHandle (must be closed)
};

namespace {

__device__ __forceinline__ void st_release_sys(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// Each warp moves whole rows  H[idx[i]] / div  into the peer's slab (16-byte stores over NVLink).
// The last CTA to finish (device-scope ticket) publishes the flag with a system-scope release.
template <bool VEC>
__global__ void __launch_bounds__(kThreads) p2p_put_rows_kernel(const float *__restrict__ H, int64_t ldh, int32_t F,
                                                               const int64_t *__restrict__ idx, int64_t k, float div,
                                                               float *remote, int64_t ldr, unsigned long long *flag,
                                                               unsigned long long flag_value,
                                                               const unsigned long long *flag_value_dev, unsigned int *ticket) {
    const int lane = threadIdx.x & 31;
    const int64_t warps_total = (int64_t)gridDim.x * kWarps;
    for (int64_t i = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); i < k; i += warps_total) {
        const int64_t r = idx ? idx[i] : i;
        const float *s = H + r * ldh;
        float *d = remote + i * ldr;
        if (VEC) {
            for (int f = lane * 4; f < F; f += 128) {
                float4 v = *reinterpret_cast<const float4 *>(s + f);
                v.x = __fdiv_rn(v.x, div); v.y = __fdiv_rn(v.y, div); v.z = __fdiv_rn(v.z, div); v.w = __fdiv_rn(v.w, div);
                *reinterpret_cast<float4 *>(d + f) = v;
            }
        } else {
            for (int f = lane; f < F; f += 32) d[f] = __fdiv_rn(s[f], div);
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int done = atomicAdd(ticket, 1u);
        if (done == gridDim.x - 1) {
            *ticket = 0;               // re-arm for the next launch on this stream
            __threadfence_system();
            st_release_sys(flag, flag_value + (flag_value_dev ? *flag_value_dev : 0ull));
        }
    }
}

__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// Bounded spin: a peer that never signals (it failed, or the schedule is wrong) must not hang the GPU.
__global__ void p2p_wait_kernel(const unsigned long long *flag, unsigned long long value,
                                const unsigned long long *value_dev, unsigned long long timeout_ns) {
    if (threadIdx.x == 0) {
        if (value_dev) value += *value_dev;
        const unsigned long long t0 = global_ns();
        while (ld_acquire_sys(flag) < value) {
            __nanosleep(64);
            if (global_ns() - t0 > timeout_ns) {
                printf("bns_p2p_wait_flag: timed out waiting for flag value %llu (have %llu)\n", value, ld_acquire_sys(flag));
                __trap();
            }
        }
    }
}

}  // namespace

namespace { void preload_exchange_kernels(); }      // fused.cuh

extern "C" int bns_p2p_create(bns_p2p_t **out, int32_t rank, int32_t world, size_t slab_bytes, int32_t n_flags) {
    BNS_REQUIRE(out, "bns_p2p_create: out is NULL");
    BNS_REQUIRE(world >= 1 && rank >= 0 && rank < world, "bns_p2p_create: bad rank/world");
    BNS_REQUIRE(n_flags >= 1, "bns_p2p_create: n_flags must be >= 1");
    bns_p2p *p = new (std::nothrow) bns_p2p();
    if (!p) return fail(BNS_E_INVALID, "bns_p2p_create: out of host memory");
    p->rank = rank; p->world = world; p->n_flags = n_flags;
    p->slab_bytes = slab_bytes ? align256(slab_bytes) : 256;
    p->peer_slab = new char *[world]();
    p->peer_flags = new unsigned long long *[world]();
    p->peer_slab_bytes = new size_t[world]();
    p->imported = new bool[world]();
    // flags block: n_flags u64 + u32 completion tickets (one per peer for bns_p2p_put_rows_f32, 16 more for the
    // all-peer puts), zero-initialised
    const size_t flag_bytes = align256((size_t)n_flags * 8) + align256((size_t)(world + 16) * 4);
    if (cudaMalloc(&p->slab, p->slab_bytes) != cudaSuccess || cudaMalloc(&p->flags, flag_bytes) != cudaSuccess) {
        int rc = fail(BNS_E_CUDA, "bns_p2p_create: cudaMalloc failed: %s", cudaGetErrorString(cudaGetLastError()));
        bns_p2p_destroy(p);
        return rc;
    }
    cudaMemset(p->slab, 0, p->slab_bytes);
    cudaMemset(p->flags, 0, flag_bytes);
    cudaDeviceSynchronize();
    p->peer_slab[rank] = p->slab;
    p->peer_flags[rank] = p->flags;
    p->peer_slab_bytes[rank] = p->slab_bytes;
    // CUDA loads a kernel's code lazily at its first launch, and that load synchronises the context: a first-ever
    // put launched while a flag wait is spinning in the same context would wait for the wait.  Load them now.
    cudaFuncAttributes fa;
    cudaFuncGetAttributes(&fa, p2p_put_rows_kernel<true>);
    cudaFuncGetAttributes(&fa, p2p_put_rows_kernel<false>);
    cudaFuncGetAttributes(&fa, p2p_wait_kernel);
    cudaFuncGetAttributes(&fa, rows_kernel<true, true>);
    cudaFuncGetAttributes(&fa, rows_kernel<false, true>);
    cudaFuncGetAttributes(&fa, rows_kernel<true, false>);
    cudaFuncGetAttributes(&fa, rows_kernel<false, false>);
    preload_exchange_kernels();
    *out = p;
    return BNS_OK;
}

extern "C" int bns_p2p_destroy(bns_p2p_t *p) {
    if (!p) return BNS_OK;
    for (int i = 0; i < p->world; ++i) {
        if (p->imported && p->imported[i]) {
            cudaIpcCloseMemHandle(p->peer_slab[i]);
            cudaIpcCloseMemHandle(p->peer_flags[i]);
        }
    }
    cudaFree(p->slab); cudaFree(p->flags);
    delete[] p->peer_slab; delete[] p->peer_flags; delete[] p->peer_slab_bytes; delete[] p->imported;
    delete p;
    return BNS_OK;
}

extern "C" int bns_p2p_local(const bns_p2p_t *p, void **slab, void **flags, size_t *slab_bytes) {
    BNS_REQUIRE(p, "bns_p2p_local: NULL handle");
    if (slab) *slab = p->slab;
    if (flags) *flags = p->flags;
    if (slab_bytes) *slab_bytes = p->slab_bytes;
    return BNS_OK;
}

extern "C" int bns_p2p_export(const bns_p2p_t *p, void *handle_out) {
    BNS_REQUIRE(p && handle_out, "bns_p2p_export: NULL argument");
    static_assert(sizeof(cudaIpcMemHandle_t) <= BNS_P2P_HANDLE_BYTES, "handle size");
    cudaIpcMemHandle_t h;
    BNS_CUDA(cudaIpcGetMemHandle(&h, p->slab));
    memcpy(handle_out, &h, sizeof(h));
    BNS_CUDA(cudaIpcGetMemHandle(&h, p->flags));
    memcpy(reinterpret_cast<char *>(handle_out) + BNS_P2P_HANDLE_BYTES, &h, sizeof(h));
    return BNS_OK;
}

extern "C" int bns_p2p_import(bns_p2p_t *p, int32_t peer, const void *handle, size_t peer_slab_bytes) {
    BNS_REQUIRE(p && handle, "bns_p2p_import: NULL argument");
    BNS_REQUIRE(peer >= 0 && peer < p->world && peer != p->rank, "bns_p2p_import: bad peer %d", peer);
    cudaIpcMemHandle_t h;
    void *ptr = nullptr;
    memcpy(&h, handle, sizeof(h));
    BNS_CUDA(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
    p->peer_slab[peer] = reinterpret_cast<char *>(ptr);
    memcpy(&h, reinterpret_cast<const char *>(handle) + BNS_P2P_HANDLE_BYTES, sizeof(h));
    BNS_CUDA(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
    p->peer_flags[peer] = reinterpret_cast<unsigned long long *>(ptr);
    p->peer_slab_bytes[peer] = peer_slab_bytes;
    p->imported[peer] = true;
    return BNS_OK;
}

extern "C" int bns_p2p_set_peer(bns_p2p_t *p, int32_t peer, void *slab, void *flags, size_t peer_slab_bytes) {
    BNS_REQUIRE(p && slab && flags, "bns_p2p_set_peer: NULL argument");
    BNS_REQUIRE(peer >= 0 && peer < p->world && peer != p->rank, "bns_p2p_set_peer: bad peer %d", peer);
    p->peer_slab[peer] = reinterpret_cast<char *>(slab);
    p->peer_flags[peer] = reinterpret_cast<unsigned long long *>(flags);
    p->peer_slab_bytes[peer] = peer_slab_bytes;
    return BNS_OK;
}

extern "C" int bns_p2p_put_rows_f32(bns_p2p_t *p, int32_t peer, size_t remote_off, int64_t ld_remote, const float *H,
                                    int64_t ldh, int64_t F, const int64_t *idx, int64_t k, float div,
                                    int32_t flag_index, uint64_t flag_value, const uint64_t *flag_value_dev,
                                    void *stream) {
    BNS_REQUIRE(p, "bns_p2p_put_rows_f32: NULL handle");
    BNS_REQUIRE(peer >= 0 && peer < p->world && peer != p->rank, "bns_p2p_put_rows_f32: bad peer %d", peer);
    BNS_REQUIRE(p->peer_slab[peer] && p->peer_flags[peer], "bns_p2p_put_rows_f32: peer %d not connected", peer);
    BNS_REQUIRE(flag_index >= 0 && flag_index < p->n_flags, "bns_p2p_put_rows_f32: bad flag index");
    BNS_REQUIRE(k >= 0 && F > 0 && ldh >= F && ld_remote >= F, "bns_p2p_put_rows_f32: bad shape");
    BNS_REQUIRE(k == 0 || div != 0.f, "bns_p2p_put_rows_f32: division by zero");   // k == 0 still publishes the flag
    BNS_REQUIRE(remote_off % 16 == 0 && remote_off + (size_t)k * ld_remote * 4 <= p->peer_slab_bytes[peer],
                "bns_p2p_put_rows_f32: remote range [%zu, +%lld rows) outside peer %d's slab (%zu bytes)", remote_off,
                (long long)k, peer, p->peer_slab_bytes[peer]);
    BNS_REQUIRE(k == 0 || H, "bns_p2p_put_rows_f32: NULL source");
    float *remote = reinterpret_cast<float *>(p->peer_slab[peer] + remote_off);
    unsigned long long *flag = p->peer_flags[peer] + flag_index;
    // ticket counters live behind the flags of THIS rank's block, one per destination peer
    unsigned int *ticket = reinterpret_cast<unsigned int *>(reinterpret_cast<char *>(p->flags) +
                                                            align256((size_t)p->n_flags * 8)) + peer;
    cudaStream_t st = as_stream(stream);
    const unsigned grid = rows_grid(k);
    if (vec_ok(H, remote, F, ldh, ld_remote))
        p2p_put_rows_kernel<true><<<grid, kThreads, 0, st>>>(H, ldh, (int32_t)F, idx, k, div, remote, ld_remote, flag,
                                                             flag_value,
                                                             reinterpret_cast<const unsigned long long *>(flag_value_dev), ticket);
    else
        p2p_put_rows_kernel<false><<<grid, kThreads, 0, st>>>(H, ldh, (int32_t)F, idx, k, div, remote, ld_remote, flag,
                                                              flag_value,
                                                              reinterpret_cast<const unsigned long long *>(flag_value_dev), ticket);
    ++g_launches;
    BNS_CUDA(cudaGetLastError());
    return BNS_OK;
}

extern "C" int bns_p2p_wait_flag(bns_p2p_t *p, int32_t flag_index, uint64_t flag_value, const uint64_t *flag_value_dev,
                                 void *stream) {
    BNS_REQUIRE(p, "bns_p2p_wait_flag: NULL handle");
    BNS_REQUIRE(flag_index >= 0 && flag_index < p->n_flags, "bns_p2p_wait_flag: bad flag index");
    p2p_wait_kernel<<<1, 32, 0, as_stream(stream)>>>(p->flags + flag_index, flag_value,
                                                     reinterpret_cast<const unsigned long long *>(flag_value_dev),
                                                     20ull * 1000000000ull);
    ++g_launches;
    BNS_CUDA(cudaGetLastError());
    return BNS_OK;
}

// =================================================================================================
// the tail of the epoch: loss, Adam, consolidated exchange, per-epoch maps, halo compaction
// =================================================================================================
#include "fused.cuh"
#include "gat.cuh"
#include "comm.cuh"

// =================================================================================================
// K8: dense layers on tcgen05 (3xTF32 with the operand split fused into the pipeline)
// =================================================================================================
#include "dense_tc.cuh"
