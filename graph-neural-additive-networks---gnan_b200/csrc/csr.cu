// Directed CSR of an edge list, built on the device by a counting sort keyed on the source (no comparison sort, no host
// round trip): replaces the COO -> scipy LIL conversion in front of the reference's Dijkstra (pre_process_datasets.py:109,129;
// batched_pyg_main.py:36-44). Neighbour order inside a row is whatever the atomics give: hop distances do not depend on it.
// Duplicate (src,dst) pairs are DETECTED (status bit 1): the reference's conversion sums them into an edge of weight 2, which
// the caller emulates by subdividing the edge (gnan_b200/preprocess.py) -- unit-weight BFS alone would be wrong there.
#include <cub/device/device_scan.cuh>

#include "common.cuh"

namespace {

__global__ void csr_degree_kernel(const int64_t *__restrict__ src, const int64_t *__restrict__ dst, int64_t E, int32_t N,
                                  int32_t *__restrict__ deg, int32_t *__restrict__ status)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    const int64_t s = src[e], d = dst[e];
    if (s < 0 || s >= N || d < 0 || d >= N) {
        atomicOr(status, 1);
        return;
    }
    atomicAdd(deg + s, 1);
}

__global__ void csr_fill_kernel(const int64_t *__restrict__ src, const int64_t *__restrict__ dst, int64_t E, int32_t N,
                                const int32_t *__restrict__ rowptr, int32_t *__restrict__ cursor, int32_t *__restrict__ col)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    const int64_t s = src[e], d = dst[e];
    if (s < 0 || s >= N || d < 0 || d >= N) return;
    col[rowptr[s] + atomicAdd(cursor + s, 1)] = (int32_t)d;
}

// any repeated neighbour in a row? Short rows (the bulk: molecules, citation graphs) are checked by ONE thread each; rows with
// more than DUP_SHORT neighbours are queued and checked by a warp each in a second, persistent kernel.
constexpr int DUP_SHORT = 16;
__global__ void csr_duplicates_short_kernel(const int32_t *__restrict__ rowptr, const int32_t *__restrict__ col, int32_t N,
                                            int32_t *__restrict__ status, int32_t *__restrict__ queue, int32_t *__restrict__ nqueue)
{
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= N) return;
    const int b = rowptr[row], deg = rowptr[row + 1] - b;
    if (deg < 2) return;
    if (deg > DUP_SHORT) {
        queue[atomicAdd(nqueue, 1)] = (int32_t)row;
        return;
    }
    int v[DUP_SHORT];
#pragma unroll
    for (int p = 0; p < DUP_SHORT; ++p) v[p] = p < deg ? col[b + p] : -1 - p;      // distinct negative fillers
    bool dup = false;
#pragma unroll
    for (int p = 0; p < DUP_SHORT; ++p)
#pragma unroll
        for (int q = p + 1; q < DUP_SHORT; ++q) dup |= v[p] == v[q];
    if (dup) atomicOr(status, 2);
}

__global__ void csr_duplicates_long_kernel(const int32_t *__restrict__ rowptr, const int32_t *__restrict__ col,
                                           const int32_t *__restrict__ queue, const int32_t *__restrict__ nqueue,
                                           int32_t *__restrict__ status)
{
    const int lane = threadIdx.x & 31;
    const int nq = *nqueue;
    const int nw = (int)((gridDim.x * blockDim.x) >> 5);
    for (int w = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5); w < nq; w += nw) {
        const int row = queue[w];
        const int b = rowptr[row], e = rowptr[row + 1];
        bool dup = false;
        for (int p = b; p < e && !dup; ++p) {
            const int v = col[p];
            for (int q = p + 1 + lane; q < e; q += 32) dup |= col[q] == v;
        }
        if (__any_sync(0xffffffffu, dup) && lane == 0) atomicOr(status, 2);
    }
}

// edge list of a batch of small graphs from its compact transfer form: endpoints as uint8 (or int16) indices inside their graph,
// the graph of edge e found by a binary search in the per-graph edge offsets (B + 1 int32 values: L1 / L2 resident)
template <typename IT>
__global__ void edges_from_local_kernel(const IT *__restrict__ src, const IT *__restrict__ dst,
                                        const int32_t *__restrict__ edge_off, const int32_t *__restrict__ node_off, int32_t B, int64_t E,
                                        int64_t *__restrict__ out)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    int lo = 0, hi = B;                                   // largest g with edge_off[g] <= e
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(edge_off + mid) <= e) lo = mid; else hi = mid;
    }
    const int64_t base = __ldg(node_off + lo);
    out[e] = base + src[e];
    out[E + e] = base + dst[e];
}

template <typename IT>
int edges_from_local(const char *who, const IT *src, const IT *dst, const int32_t *edge_off, const int32_t *node_off, int32_t B, int64_t E,
                     int64_t *edge_index, gnan_stream_t stream)
{
    GNAN_REQUIRE(B >= 0 && E >= 0, "%s: negative sizes", who);
    GNAN_REQUIRE(E == 0 || (B > 0 && src && dst && edge_off && node_off && edge_index), "%s: NULL pointer", who);
    if (E) {
        edges_from_local_kernel<IT><<<(unsigned)ceil_div64(E, 256), 256, 0, (cudaStream_t)stream>>>(src, dst, edge_off, node_off, B, E,
                                                                                                  edge_index);
        GNAN_LAUNCH_OK();
    }
    return GNAN_OK;
}

}  // namespace

extern "C" int gnan_edges_from_local(const uint8_t *src, const uint8_t *dst, const int32_t *edge_off, const int32_t *node_off, int32_t B,
                                     int64_t E, int64_t *edge_index, gnan_stream_t stream)
{
    return edges_from_local("edges_from_local", src, dst, edge_off, node_off, B, E, edge_index, stream);
}

extern "C" int gnan_edges_from_local_i16(const int16_t *src, const int16_t *dst, const int32_t *edge_off, const int32_t *node_off,
                                         int32_t B, int64_t E, int64_t *edge_index, gnan_stream_t stream)
{
    return edges_from_local("edges_from_local_i16", src, dst, edge_off, node_off, B, E, edge_index, stream);
}

extern "C" size_t gnan_build_csr_workspace_bytes(int32_t N, int64_t E)
{
    size_t scan = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, scan, (const int32_t *)nullptr, (int32_t *)nullptr, N + 1);
    return (scan + 255) / 256 * 256 + sizeof(int32_t) * ((size_t)N + 1) * 2;
}

extern "C" int gnan_build_csr(const int64_t *src, const int64_t *dst, int64_t E, int32_t N, int32_t *rowptr, int32_t *col,
                              int32_t *status, void *workspace, size_t workspace_bytes, gnan_stream_t stream)
{
    GNAN_REQUIRE(N >= 0 && E >= 0 && rowptr && status, "build_csr: bad arguments");
    GNAN_REQUIRE(E == 0 || (src && dst && col), "build_csr: NULL edge arrays");
    GNAN_REQUIRE(E < ((int64_t)1 << 31), "build_csr: more than 2^31 - 1 edges");
    const size_t need = gnan_build_csr_workspace_bytes(N, E);
    if (!workspace || workspace_bytes < need) {
        gnan_set_error("build_csr: workspace %zu < %zu bytes", workspace_bytes, need);
        return GNAN_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    size_t scan = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, scan, (const int32_t *)nullptr, (int32_t *)nullptr, N + 1);
    const size_t scan_al = (scan + 255) / 256 * 256;
    int32_t *deg = (int32_t *)((uint8_t *)workspace + scan_al);        // [N+1] (last entry stays 0)
    int32_t *cursor = deg + (N + 1);                                   // [N+1]
    GNAN_CUDA(cudaMemsetAsync(deg, 0, sizeof(int32_t) * ((size_t)N + 1) * 2, st));
    GNAN_CUDA(cudaMemsetAsync(status, 0, sizeof(int32_t), st));
    if (E) {
        csr_degree_kernel<<<(unsigned)ceil_div64(E, 256), 256, 0, st>>>(src, dst, E, N, deg, status);
        GNAN_LAUNCH_OK();
    }
    GNAN_CUDA(cub::DeviceScan::ExclusiveSum(workspace, scan, deg, rowptr, N + 1, st));
    gnan_count_launch();
    if (E) {
        csr_fill_kernel<<<(unsigned)ceil_div64(E, 256), 256, 0, st>>>(src, dst, E, N, rowptr, cursor, col);
        GNAN_LAUNCH_OK();
        // deg[] is free after the scan: it becomes the queue of long rows; cursor[N] (never touched by the fill) is its length
        csr_duplicates_short_kernel<<<(unsigned)ceil_div64(N, 256), 256, 0, st>>>(rowptr, col, N, status, deg, cursor + N);
        GNAN_LAUNCH_OK();
        csr_duplicates_long_kernel<<<2 * gnan_sm_count(), 256, 0, st>>>(rowptr, col, deg, cursor + N, status);
        GNAN_LAUNCH_OK();
    }
    return GNAN_OK;
}
