// All-pairs hop distances on the GPU (multi-source BFS) and the reference-format converters.
//
// Reference lines replaced: pre_process_datasets.py:109-121 / :128-140 (scipy dijkstra on unit weights + the per-element
// Python normaliser loop) and batched_pyg_main.py:36-44 (networkx BFS per node).
// Output: uint8 hop matrix (level, 255 = unreachable) and int32 level sizes cnt[i,d]; the reference's two fp32 [N,N]
// matrices are node_distances = 1/(1+hop) and normalization_matrix = cnt[i, hop[i,j]] (gnan_hops_to_reference).
#include <algorithm>
#include <type_traits>
#include "common.cuh"

namespace {

// ---- batched small graphs, v3: a GROUP of 4 warps per graph slot, bit-parallel over SOURCES -----------------------------------
// A lane owns ONE vertex v and keeps the bitmask of sources that reach it (W = ceil(n/32) words). Level L is a pull over v's
// out-neighbours u: new[v] = (OR_u frontier[u]) & ~visited[v]; a new bit s means dist(v -> s) = L, i.e. hop[v][s] = L, and
// popc(new[v]) is row v's level-L count (no atomics). One warp per graph would be bound by the latency of its dependent
// instruction stream (a lane walking up to 4 vertices one after the other), so the warps of a group advance a level together
// (named barrier with an OR reduction = "did anybody reach a new vertex"): graphs of 65..128 nodes take the 4 warps of a group,
// graphs of 33..64 nodes run two at a time on warp pairs, graphs of up to 32 nodes four at a time on single warps, each in its
// share of the group's shared-memory slice.
// The n x n hop block is assembled in shared memory (byte stores there), padded so that it is congruent to its global address
// mod 16, and leaves as 16-byte vector stores: the global hop bytes are written exactly once, unreachable pairs included (no
// memset). The level counts (<= 127 per entry) are collected in a uint8 [n][nbins] shared-memory table and leave as one
// coalesced int32 block per graph, zeros included: no memset of the level table and no scattered 4-byte global stores per
// (vertex, level), which cost a 32-byte sector each.
constexpr int BV3_MAX_W = 4;                               // up to 128 nodes per graph
constexpr int BV3_GW = 4;                                  // warps per group
constexpr int BV3_MAX_GROUPS = 5;                          // groups per CTA (3 named barriers each: ids 1..15)

__host__ __device__ inline size_t round16(size_t x) { return (x + 15) / 16 * 16; }
__host__ __device__ inline size_t bv3_hop_bytes(int cap) { return round16((size_t)cap * cap + 16); }
__host__ __device__ constexpr int bv3_ws(int W) { return W == 3 ? 4 : W; }         // frontier row stride in words: 16-byte rows for W = 3
// two frontier buffers [n][WS] (+ the adjacency bit matrix [n][WS] when the kernel builds it from the edge segment itself)
__host__ __device__ inline size_t bv3_fr_bytes(int cap, int W, bool local = false)
{
    return round16((size_t)(local ? 3 : 2) * cap * bv3_ws(W) * 4);
}

// frontier rows move as ONE shared-memory access (LDS.128 / LDS.64 instead of W scalar loads per neighbour)
template <int W>
__device__ __forceinline__ void bv3_or_row(const uint32_t *row, uint32_t (&acc)[W])
{
    if (W >= 3) {
        const uint4 q = *reinterpret_cast<const uint4 *>(row);
        acc[0] |= q.x; acc[1] |= q.y; acc[2] |= q.z;
        if (W == 4) acc[W - 1] |= q.w;
    } else if (W == 2) {
        const uint2 q = *reinterpret_cast<const uint2 *>(row);
        acc[0] |= q.x; acc[1] |= q.y;
    } else {
        acc[0] |= row[0];
    }
}
template <int W>
__device__ __forceinline__ void bv3_store_row(uint32_t *row, const uint32_t (&w)[W])
{
    if (W >= 3) *reinterpret_cast<uint4 *>(row) = make_uint4(w[0], w[1], w[2], W == 4 ? w[W - 1] : 0u);
    else if (W == 2) *reinterpret_cast<uint2 *>(row) = make_uint2(w[0], w[1]);
    else row[0] = w[0];
}
__host__ __device__ inline size_t bv3_need(int cap, int W, int nbins, bool levels, bool local = false)
{
    return bv3_hop_bytes(cap) + bv3_fr_bytes(cap, W, local) + (levels ? round16((size_t)cap * nbins) : 0);
}

// up to 8 out-neighbours of a vertex travel with it as bytes of two registers (lo, hi), dg of them
__device__ __forceinline__ void bv3_keep(uint32_t &lo, uint32_t &hi, int &dg, uint32_t u)
{
    const int sh = 8 * (dg & 3);
    if (dg < 4) lo = (lo & ~(0xffu << sh)) | (u << sh);
    else hi = (hi & ~(0xffu << sh)) | (u << sh);
    ++dg;
}
// LOCAL: the out-neighbours of a vertex from its adjacency row; more than 8: many = 1 and the level loop walks the row instead
template <int W>
__device__ __forceinline__ void bv3_local_nbrs(const uint32_t *arow, uint32_t &lo, uint32_t &hi, int &dg, int &many)
{
    int deg = 0;
#pragma unroll
    for (int ww = 0; ww < W; ++ww) deg += __popc(arow[ww]);
    if (deg <= 8) {
#pragma unroll
        for (int ww = 0; ww < W; ++ww) {
            uint32_t m = arow[ww];
            while (m) {
                bv3_keep(lo, hi, dg, (uint32_t)(ww * 32 + __ffs(m) - 1));
                m &= m - 1;
            }
        }
    } else {
        many = 1;
    }
}
// acc |= the frontier rows fc [n][WS] of the dg kept neighbours
template <int W>
__device__ __forceinline__ void bv3_pull_kept(const uint32_t *fc, uint32_t lo, uint32_t hi, int dg, uint32_t (&acc)[W])
{
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        if (t < dg) {
            const uint32_t u = ((t < 4 ? lo : hi) >> (8 * (t & 3))) & 0xffu;
            bv3_or_row<W>(fc + u * bv3_ws(W), acc);
        }
    }
}
// acc |= the frontier rows of every neighbour in the adjacency row arow (rows with more than 8 neighbours)
template <int W>
__device__ __forceinline__ void bv3_pull_row(const uint32_t *fc, const uint32_t *arow, uint32_t (&acc)[W])
{
#pragma unroll
    for (int ww = 0; ww < W; ++ww) {
        uint32_t m = arow[ww];
        while (m) {
            bv3_or_row<W>(fc + (ww * 32 + __ffs(m) - 1) * bv3_ws(W), acc);
            m &= m - 1;
        }
    }
}

template <int G>
__device__ __forceinline__ void bv3_sync(int bar)
{
    if (G == 1) __syncwarp();
    else asm volatile("barrier.sync %0, %1;" :: "r"(bar), "n"(32 * G) : "memory");
}

template <int G>
__device__ __forceinline__ bool bv3_any(int bar, bool p)
{
    if (G == 1) {
        __syncwarp();
        return __any_sync(0xffffffffu, p);
    }
    uint32_t r;
    asm volatile("{\n\t.reg .pred pi, po;\n\tsetp.ne.u32 pi, %3, 0;\n\tbarrier.red.or.pred po, %1, %2, pi;\n\tselp.u32 %0, 1, 0, po;\n\t}"
                 : "=r"(r) : "r"(bar), "n"(32 * G), "r"((uint32_t)p) : "memory");
    return r != 0;
}

// one graph on G warps, W = ceil(n/32) <= G words per vertex; thread ts = wsub * 32 + lane owns vertex ts.
// LOCAL: the out-neighbours come from the adjacency bit matrix adj [n][WS] in shared memory (built by bv3_run from the graph's own
// edge segment) instead of the CSR. The hop bytes of a level are scattered two bits per step (lowest and highest new source).
template <int W, int G, bool LOCAL>
__device__ __forceinline__ int bv3_graph(const int32_t *__restrict__ rowptr, const int32_t *__restrict__ col, int n0, int n, int ts,
                                         int bar, uint8_t *hb, uint32_t *frs, const uint32_t *adj, uint8_t *cs, int nbins, bool levels,
                                         int32_t *overflow)
{
    constexpr int WS = bv3_ws(W);
    const int v = ts, lane = ts & 31, wsub = ts >> 5;
    const bool mine = v < n;
    uint32_t vis[W], nb_lo = 0xffffffffu, nb_hi = 0xffffffffu;
    int dg = 0, e8 = 0, e1 = 0;
#pragma unroll
    for (int ww = 0; ww < W; ++ww) vis[ww] = 0u;
    if (mine) {
        if (LOCAL) {
            bv3_local_nbrs<W>(adj + v * WS, nb_lo, nb_hi, dg, e1);  // e1 = 1: more than 8 neighbours
        } else {
            const int eb = rowptr[n0 + v], ee = rowptr[n0 + v + 1];
            int e = eb;
            for (; e < ee && dg < 8; ++e) {                          // neighbours outside the graph are ignored
                const int u = __ldg(col + e) - n0;
                if (u >= 0 && u < n) bv3_keep(nb_lo, nb_hi, dg, (uint32_t)u);
            }
            e8 = e; e1 = ee;
        }
#pragma unroll
        for (int ww = 0; ww < W; ++ww) vis[ww] = ww == wsub ? 1u << lane : 0u;
        bv3_store_row<W>(frs + v * WS, vis);
        hb[v * n + v] = 0;
        if (levels) cs[v * nbins] = 1;
    }
    bv3_sync<G>(bar);
    int lvl_max = 0;
    for (int level = 1; level <= n; ++level) {
        const uint32_t *fc = frs + ((level - 1) & 1) * n * WS;
        uint32_t *fn = frs + (level & 1) * n * WS;
        const uint8_t lv = (uint8_t)min(level, 254);
        bool any = false;
        if (mine) {
            uint32_t acc[W];
#pragma unroll
            for (int ww = 0; ww < W; ++ww) acc[ww] = 0u;
            bv3_pull_kept<W>(fc, nb_lo, nb_hi, dg, acc);
            if (LOCAL) {
                if (e1) bv3_pull_row<W>(fc, adj + v * WS, acc);      // rows with more than 8 neighbours
            } else {
                for (int e = e8; e < e1; ++e) {                      // rows with more than 8 neighbours
                    const int u = __ldg(col + e) - n0;
                    if (u >= 0 && u < n) bv3_or_row<W>(fc + u * WS, acc);
                }
            }
            int newc = 0;
#pragma unroll
            for (int ww = 0; ww < W; ++ww) {
                acc[ww] &= ~vis[ww];
                vis[ww] |= acc[ww];
                newc += __popc(acc[ww]);
            }
            bv3_store_row<W>(fn + v * WS, acc);
#pragma unroll
            for (int ww = 0; ww < W; ++ww) {
                uint32_t m = acc[ww];
                uint8_t *rowp = hb + v * n + ww * 32;
                while (m) {
                    const int lo = __ffs(m) - 1, hi = 31 - __clz(m);
                    rowp[lo] = lv;
                    rowp[hi] = lv;
                    m &= m - 1;
                    m &= ~(1u << hi);
                }
            }
            if (newc) {
                any = true;
                if (level > 254 || level >= nbins - 1) atomicExch(overflow, 1);
                else if (levels) cs[v * nbins + level] = (uint8_t)newc;
            }
        }
        if (!bv3_any<G>(bar, any)) break;
        lvl_max = level;
    }
    int reached = 0;
#pragma unroll
    for (int ww = 0; ww < W; ++ww) reached += __popc(vis[ww]);
    if (levels && mine) cs[v * nbins + nbins - 1] = (uint8_t)(n - reached);
    return lvl_max;
}

// graphs by size class, one thread per graph, warp-aggregated counters: classes 0..3 by word count (0 = 97..128 nodes ... 3 = up
// to 32) for the v3 kernel, class 4 = more than 128 nodes for apsp_batched_large_kernel. cls[0..4) = the sizes of classes 0..3,
// cls[4 + c * B ...) = the graphs of class c in arbitrary order; class 4 has its size at cls[4 * B + 4] and its graphs from
// cls[4 * B + 5] on. The caller zeroes the size words. A batch without graphs of more than 128 nodes leaves class 4 empty and has
// nothing written at or beyond cls[4 * B + 4] (order_ws [4 * B + 4]).
// The v3 kernel walks the classes largest first: the expensive graphs start first, and the groups of a CTA run the same
// instantiation of bv3_graph side by side (the instantiations do not fit the instruction cache together).
__global__ void bv3_classify_kernel(const int32_t *__restrict__ node_off, int B, int32_t *__restrict__ cls)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    const bool ok = b < B;
    int c = 5;                                                            // (no graph: a value of no class)
    if (ok) {
        const int n = node_off[b + 1] - node_off[b];
        c = n > 32 * BV3_MAX_W ? 4 : 3 - min(3, max(0, (n - 1) >> 5));
    }
    const uint32_t peers = __match_any_sync(0xffffffffu, c);
    const int lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
    int base = 0;
    if (ok && lane == leader) base = atomicAdd(cls + (c < 4 ? c : 4 + 4 * B), __popc(peers));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (ok) cls[4 + (size_t)c * B + (c >> 2) + base + __popc(peers & ((1u << lane) - 1))] = b;   // class 4: after its size word
}

template <typename IT>
struct Bv3OutT {
    uint8_t *hop;
    int32_t *cnt;
    float *rscale;
    const float *rcp_tab;
    int nbins;
    // LOCAL: the batch's edges grouped by graph, endpoints as indices inside the graph (uint8, or int16 for the fused readout);
    // *status |= 1 for an endpoint >= n (edge dropped), |= 2 for a repeated (src,dst) pair (gnan_build_csr's status bits)
    const IT *lsrc, *ldst;
    const int32_t *edge_off;
    int32_t *status;
};
using Bv3Out = Bv3OutT<uint8_t>;

// an endpoint of the transfer form as an unsigned index: a negative int16 becomes >= 32768, i.e. out of every graph's range
__device__ __forceinline__ uint32_t local_index(uint8_t x) { return x; }
__device__ __forceinline__ uint32_t local_index(int16_t x) { return (uint16_t)x; }

// graph b on the G warps of a sub-group: fill the slice, BFS, write the level table and the hop block out
template <int W, int G, bool LOCAL>
__device__ __forceinline__ int bv3_run(const int32_t *__restrict__ rowptr, const int32_t *__restrict__ col,
                                       const int32_t *__restrict__ node_off, const int64_t *__restrict__ hop_off, int64_t b, int cap,
                                       int ts, int bar, uint8_t *slice, const Bv3Out &o, bool levels, int32_t *overflow)
{
    constexpr int T = 32 * G;
    const int n0 = node_off[b], n = node_off[b + 1] - n0, nbins = o.nbins;
    uint8_t *gb = o.hop + hop_off[b];
    const int pad = (int)(reinterpret_cast<uintptr_t>(gb) & 15);
    uint8_t *hb = slice + pad;                                                  // hb + k  ==  gb + k  (mod 16)
    constexpr int WS = bv3_ws(W);
    uint32_t *frs = reinterpret_cast<uint32_t *>(slice + bv3_hop_bytes(cap));  // [2][n][WS] (+ adjacency [n][WS])
    uint32_t *adj = frs + 2 * n * WS;
    uint8_t *cs = slice + bv3_hop_bytes(cap) + bv3_fr_bytes(cap, W, LOCAL);   // [n][nbins]
    const int total = n * n;
    for (int t = ts * 16; t < total + 16; t += T * 16)
        *reinterpret_cast<uint4 *>(slice + t) = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
    if (levels)
        for (int t = ts * 16; t < n * nbins; t += T * 16) *reinterpret_cast<uint4 *>(cs + t) = make_uint4(0u, 0u, 0u, 0u);
    if (LOCAL) {
        for (int t = ts; t < n * WS; t += T) adj[t] = 0u;
        bv3_sync<G>(bar);
        const int e0 = o.edge_off[b], e1 = o.edge_off[b + 1];
        int flags = 0;
        for (int e = e0 + ts; e < e1; e += T) {
            const uint32_t s = o.lsrc[e], d = o.ldst[e];
            if (s < (uint32_t)n && d < (uint32_t)n) {
                const uint32_t bit = 1u << (d & 31);
                if (atomicOr(adj + s * WS + (d >> 5), bit) & bit) flags |= 2;
            } else {
                flags |= 1;
            }
        }
        if (flags) atomicOr(o.status, flags);
    }
    bv3_sync<G>(bar);
    const int lm = bv3_graph<W, G, LOCAL>(rowptr, col, n0, n, ts, bar, hb, frs, adj, cs, nbins, levels, overflow);
    bv3_sync<G>(bar);
    if (levels) {
        const int nt = n * nbins;                                               // the graph's [n][nbins] block is contiguous
        const bool vec_tab = (nbins & 3) == 0;
        if (o.cnt) {
            int32_t *gc = o.cnt + (int64_t)n0 * nbins;
            if (vec_tab) {
                for (int t = ts * 4; t < nt; t += T * 4) {
                    const uint32_t c4 = *reinterpret_cast<const uint32_t *>(cs + t);
                    *reinterpret_cast<int4 *>(gc + t) = make_int4(c4 & 0xff, (c4 >> 8) & 0xff, (c4 >> 16) & 0xff, c4 >> 24);
                }
            } else {
                for (int t = ts; t < nt; t += T) gc[t] = cs[t];
            }
        }
        if (o.rscale) {                              // 1/count (0 for empty levels): gnan_level_rscale fused
            float *gr = o.rscale + (int64_t)n0 * nbins;
            if (vec_tab) {
                for (int t = ts * 4; t < nt; t += T * 4) {
                    const uint32_t c4 = *reinterpret_cast<const uint32_t *>(cs + t);
                    *reinterpret_cast<float4 *>(gr + t) = make_float4(o.rcp_tab[c4 & 0xff], o.rcp_tab[(c4 >> 8) & 0xff],
                                                                      o.rcp_tab[(c4 >> 16) & 0xff], o.rcp_tab[c4 >> 24]);
                }
            } else {
                for (int t = ts; t < nt; t += T) gr[t] = o.rcp_tab[cs[t]];
            }
        }
    }
    // copy out: head bytes up to the first 16-byte boundary, vector body, tail bytes
    const int head = min(total, (16 - pad) & 15);
    if (ts < head) gb[ts] = hb[ts];
    const int body = (total - head) / 16;
    for (int t = ts; t < body; t += T)
        *reinterpret_cast<uint4 *>(gb + head + t * 16) = *reinterpret_cast<const uint4 *>(hb + head + t * 16);
    const int tail0 = head + body * 16;
    if (ts < 16 && tail0 + ts < total) gb[tail0 + ts] = hb[tail0 + ts];
    return lm;
}

// ---- the batched BFS fused with the output-normalised graph readout (LOCAL edges; models.py:366-384) -------------------------
// agg_bd_graph_fwd_kernel (csrc/agg_bd.cu) computes out / colw / Q from the hop bytes and the normaliser table that the BFS wrote.
// Here the BFS folds the pair statistics P[j,d] = sum_{i: hop(i,j) = d} 1/count(i,d) straight into them, level by level:
// colw[j,c'] += T[d,c'] P[j,d] in lane j's registers, Q[b,d,c] += S[j,c] P[j,d] as one warp sum per level into the warp's own
// [nbins][C] slot of shared memory (the slots are added in warp order at the end: no float atomics, fixed order). Neither hop
// bytes, nor a level table, nor P reach global memory. P[.,d] after the barrier of level d, summed over i in ascending order:
// on a symmetric graph the i at distance d from j are j's own new sources of the level, and count(i,d) is i's popcount (rcl,
// published by every lane before the barrier); on a directed graph lane j walks the new-frontier rows of all n vertices for
// bit j instead (slower, same result). Levels >= nbins-1 only set the overflow flag (the level table's contract).
struct Bv3Readout {
    const float *T;      // [nbins][Cr]
    const float *S;      // [sumN][C]
    int Cr, C;
    float *out, *colw, *Q;   // [B][C], [sumN][Cr], [B][nbins][C]
};

// frontier rows [2][cap][WS], adjacency [cap][WS], 1/count [2][cap], per-warp Q [G][nbins][CC] + per-warp out [G][CC]
__host__ __device__ inline size_t bv3_ro_need(int cap, int W, int G, int nbins, int CC)
{
    return round16((size_t)3 * cap * bv3_ws(W) * 4 + (size_t)2 * cap * 4 + (size_t)G * (nbins + 1) * CC * 4);
}

// lane's share of bin d: colw += T[d,:] p, the warp's Q slot [d,:] = sum over the warp's lanes of S[v,:] p (all 32 lanes call it)
template <int CC>
__device__ __forceinline__ void bv3_ro_fold(int d, float p, const float (&s)[CC], float (&cw)[CC], float *sqw, const Bv3Readout &r,
                                            int lane)
{
#pragma unroll
    for (int c = 0; c < CC; ++c) {
        if (c < r.Cr) cw[c] = fmaf(__ldg(r.T + d * r.Cr + c), p, cw[c]);
        if (c < r.C) {
            float q = s[c] * p;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
            if (lane == 0) sqw[d * CC + c] = q;
        }
    }
}

template <int W, int G, int CC, typename IT>
__device__ __forceinline__ int bv3_readout_run(const int32_t *__restrict__ node_off, int64_t b, int ts, int bar, uint8_t *slice,
                                               const Bv3OutT<IT> &o, const Bv3Readout &r, int32_t *overflow)
{
    constexpr int T = 32 * G, WS = bv3_ws(W);
    const int n0 = node_off[b], n = node_off[b + 1] - n0, nbins = o.nbins, nq = nbins * CC;
    const int v = ts, lane = ts & 31, wsub = ts >> 5;
    const bool mine = v < n;
    uint32_t *frs = reinterpret_cast<uint32_t *>(slice);                       // [2][n][WS]
    uint32_t *adj = frs + 2 * n * WS;                                          // [n][WS]
    float *rcl = reinterpret_cast<float *>(adj + n * WS);                      // [2][n] 1/count of the current level (by parity)
    float *sq = rcl + 2 * n, *so = sq + G * nq;                                // [G][nbins][CC], [G][CC]
    float *sqw = sq + wsub * nq;
    for (int t = ts; t < n * WS; t += T) adj[t] = 0u;
    for (int t = ts; t < G * (nq + CC); t += T) sq[t] = 0.f;
    bv3_sync<G>(bar);
    const int e0 = o.edge_off[b], e1 = o.edge_off[b + 1];
    int flags = 0;                                                             // status bits as gnan_apsp_bfs_batched_local
    for (int e = e0 + ts; e < e1; e += T) {
        const uint32_t s = local_index(o.lsrc[e]), d = local_index(o.ldst[e]);
        if (s < (uint32_t)n && d < (uint32_t)n) {
            const uint32_t bit = 1u << (d & 31);
            if (atomicOr(adj + s * WS + (d >> 5), bit) & bit) flags |= 2;
        } else {
            flags |= 1;
        }
    }
    if (flags) atomicOr(o.status, flags);
    bv3_sync<G>(bar);
    bool asym = false;
    for (int e = e0 + ts; e < e1; e += T) {
        const uint32_t s = local_index(o.lsrc[e]), d = local_index(o.ldst[e]);
        if (s < (uint32_t)n && d < (uint32_t)n && !((adj[d * WS + (s >> 5)] >> (s & 31)) & 1u)) asym = true;
    }
    const bool sym = !bv3_any<G>(bar, asym);

    float s[CC], cw[CC];
#pragma unroll
    for (int c = 0; c < CC; ++c) {
        s[c] = (mine && c < r.C) ? r.S[(int64_t)(n0 + v) * r.C + c] : 0.f;
        cw[c] = 0.f;
    }
    uint32_t vis[W], nb_lo = 0xffffffffu, nb_hi = 0xffffffffu;
    int dg = 0, many = 0;
#pragma unroll
    for (int ww = 0; ww < W; ++ww) vis[ww] = 0u;
    if (mine) {
        bv3_local_nbrs<W>(adj + v * WS, nb_lo, nb_hi, dg, many);
#pragma unroll
        for (int ww = 0; ww < W; ++ww) vis[ww] = ww == wsub ? 1u << lane : 0u;
        bv3_store_row<W>(frs + v * WS, vis);
    }
    bv3_ro_fold<CC>(0, mine ? 1.f : 0.f, s, cw, sqw, r, lane);                 // level 0: v itself, count 1
    bv3_sync<G>(bar);
    int lvl_max = 0;
    for (int level = 1; level <= n; ++level) {
        const uint32_t *fc = frs + ((level - 1) & 1) * n * WS;
        uint32_t *fn = frs + (level & 1) * n * WS;
        float *rc = rcl + (level & 1) * n;
        bool any = false;
        uint32_t nw[W];
        if (mine) {
#pragma unroll
            for (int ww = 0; ww < W; ++ww) nw[ww] = 0u;
            bv3_pull_kept<W>(fc, nb_lo, nb_hi, dg, nw);
            if (many) bv3_pull_row<W>(fc, adj + v * WS, nw);
            int newc = 0;
#pragma unroll
            for (int ww = 0; ww < W; ++ww) {
                nw[ww] &= ~vis[ww];
                vis[ww] |= nw[ww];
                newc += __popc(nw[ww]);
            }
            bv3_store_row<W>(fn + v * WS, nw);
            rc[v] = newc ? __frcp_rn((float)newc) : 0.f;
            if (newc) {
                any = true;
                if (level >= nbins - 1) atomicExch(overflow, 1);
            }
        }
        if (!bv3_any<G>(bar, any)) break;
        lvl_max = level;
        float p = 0.f;                                                         // P[v, level]
        if (mine) {
            if (sym) {                      // v's new sources (one channel: reloaded from fn, 5 groups per CTA fit 48 registers)
#pragma unroll
                for (int ww = 0; ww < W; ++ww) {
                    uint32_t m = CC == 1 ? fn[v * WS + ww] : nw[ww];
                    while (m) {
                        p += rc[ww * 32 + __ffs(m) - 1];
                        m &= m - 1;
                    }
                }
            } else {
                for (int i = 0; i < n; ++i)
                    if ((fn[i * WS + wsub] >> lane) & 1u) p += rc[i];
            }
        }
        if (level < nbins - 1) bv3_ro_fold<CC>(level, p, s, cw, sqw, r, lane);
    }
    // unreachable bin: sum over the i that do not reach v of 1/(i's unreachable count); skipped for connected graphs
    int reached = 0;
#pragma unroll
    for (int ww = 0; ww < W; ++ww) reached += __popc(vis[ww]);
    if (bv3_any<G>(bar, mine && reached < n)) {                                // (both frontier / 1/count buffers are free now)
        if (mine) {
            rcl[v] = reached < n ? __frcp_rn((float)(n - reached)) : 0.f;
            if (!sym) bv3_store_row<W>(frs + v * WS, vis);
        }
        bv3_sync<G>(bar);
        float U = 0.f;
        if (mine) {
            if (sym) {
#pragma unroll
                for (int ww = 0; ww < W; ++ww) {
                    const int left = n - ww * 32;
                    uint32_t m = ~vis[ww] & (left >= 32 ? 0xffffffffu : (left > 0 ? (1u << left) - 1u : 0u));
                    while (m) {
                        U += rcl[ww * 32 + __ffs(m) - 1];
                        m &= m - 1;
                    }
                }
            } else {
                for (int i = 0; i < n; ++i)
                    if (!((frs[i * WS + wsub] >> lane) & 1u)) U += rcl[i];
            }
        }
        bv3_ro_fold<CC>(nbins - 1, U, s, cw, sqw, r, lane);
    }
    if (mine) {
#pragma unroll
        for (int c = 0; c < CC; ++c)
            if (c < r.Cr) r.colw[(int64_t)(n0 + v) * r.Cr + c] = cw[c];
    }
    // out[b,c] = sum_v S[v,c] colw[v,c']: a warp sum each, then the warps in order
#pragma unroll
    for (int c = 0; c < CC; ++c) {
        if (c < r.C) {
            float q = s[c] * cw[r.Cr == 1 ? 0 : c];
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) q += __shfl_xor_sync(0xffffffffu, q, off);
            if (lane == 0) so[wsub * CC + c] = q;
        }
    }
    bv3_sync<G>(bar);
    for (int t = ts; t < nbins * r.C; t += T) {                                // Q[b] in full (empty bins: 0), coalesced
        const int d = t / r.C, c = t - d * r.C;
        float q = 0.f;
#pragma unroll
        for (int w = 0; w < G; ++w) q += sq[w * nq + d * CC + c];
        r.Q[(int64_t)b * nbins * r.C + t] = q;
    }
    if (ts < r.C) {
        float q = 0.f;
#pragma unroll
        for (int w = 0; w < G; ++w) q += so[w * CC + ts];
        r.out[b * r.C + ts] = q;
    }
    return lvl_max;
}

// one work item of the v3 kernel: the BFS of bv3_run, or (CC > 0) the BFS fused with the graph readout
template <int W, int G, bool LOCAL, int CC, typename IT>
__device__ __forceinline__ int bv3_item(const int32_t *__restrict__ rowptr, const int32_t *__restrict__ col,
                                        const int32_t *__restrict__ node_off, const int64_t *__restrict__ hop_off, int64_t b, int cap,
                                        int ts, int bar, uint8_t *slice, const Bv3OutT<IT> &o, const Bv3Readout &r, bool levels,
                                        int32_t *overflow)
{
    if constexpr (CC > 0) return bv3_readout_run<W, G, CC, IT>(node_off, b, ts, bar, slice, o, r, overflow);
    else return bv3_run<W, G, LOCAL>(rowptr, col, node_off, hop_off, b, cap, ts, bar, slice, o, levels, overflow);
}

// the batch's edge list in its transfer form (LOCAL instantiation: no CSR; rowptr / col are NULL); IT = int16 only with CC > 0
template <typename IT>
struct Bv3EdgesT {
    const IT *src, *dst;
    const int32_t *edge_off;
    int32_t *status;
};
using Bv3Edges = Bv3EdgesT<uint8_t>;

// order = the output of bv3_classify_kernel
// (the multi-channel readout instantiations keep the level's new bits across the barrier: 4 groups per CTA give them 64 registers)
constexpr int bv3_max_groups(int cc) { return cc > 1 ? BV3_MAX_GROUPS - 1 : BV3_MAX_GROUPS; }
template <bool LOCAL, int CC = 0, typename IT = uint8_t>
__global__ void __launch_bounds__(32 * BV3_GW * bv3_max_groups(CC), 2)
apsp_batched_v3_kernel(const int32_t *__restrict__ rowptr, const int32_t *__restrict__ col, const int32_t *__restrict__ node_off,
                       const int64_t *__restrict__ hop_off, int B, int max_n, int groups_per_cta, int slice_bytes, uint8_t *__restrict__ hop,
                       int32_t *__restrict__ cnt, float *__restrict__ rscale, int nbins, int32_t *__restrict__ overflow,
                       int32_t *__restrict__ max_level, const int32_t *__restrict__ order, Bv3EdgesT<IT> le, Bv3Readout ro)
{
    extern __shared__ __align__(16) uint8_t sm3[];
    __shared__ float rcp_tab[256];
    const bool levels = cnt != nullptr || rscale != nullptr;
    if (rscale) {
        for (int t = threadIdx.x; t < 256; t += blockDim.x) rcp_tab[t] = t > 0 ? 1.0f / (float)t : 0.f;   // as level_rscale_kernel
        __syncthreads();
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = warp / BV3_GW, wq = warp % BV3_GW;
    uint8_t *gslice = sm3 + (size_t)g * slice_bytes;
    const int bar_group = 1 + 3 * g;
    const Bv3OutT<IT> out{hop, cnt, rscale, rcp_tab, nbins, le.src, le.dst, le.edge_off, le.status};
    const int c0 = order[0], c_big = c0 + order[1], c2 = order[2], c3 = order[3];
    const int32_t *ord0 = order + 4, *ord1 = ord0 + B, *ord2 = ord1 + B, *ord3 = ord2 + B;
    const int items2 = (c2 + 1) / 2, items1 = (c3 + 3) / 4;
    const int64_t n_items = (int64_t)c_big + items2 + items1, stride = (int64_t)gridDim.x * groups_per_cta;
    const int cap2 = min(max_n, 64), cap1 = min(max_n, 32);
    const int half = (slice_bytes / 2) & ~15, quarter = (slice_bytes / 4) & ~15;
    int lvl_max = 0;
    for (int64_t t = (int64_t)blockIdx.x * groups_per_cta + g; t < n_items; t += stride) {
        if (t < c_big) {                                             // 65..128 nodes: the whole group
            const int64_t b = t < c0 ? ord0[t] : ord1[t - c0];
            const int n = node_off[b + 1] - node_off[b];
            const int ts = wq * 32 + lane;
            const int lm = n <= 96 ? bv3_item<3, 4, LOCAL, CC, IT>(rowptr, col, node_off, hop_off, b, max_n, ts, bar_group, gslice, out, ro, levels, overflow)
                                   : bv3_item<4, 4, LOCAL, CC, IT>(rowptr, col, node_off, hop_off, b, max_n, ts, bar_group, gslice, out, ro, levels, overflow);
            lvl_max = max(lvl_max, lm);
        } else if (t < c_big + items2) {                             // 33..64 nodes: two graphs on the two warp pairs
            const int pr = wq >> 1;
            const int64_t idx = 2 * (t - c_big) + pr;
            if (idx < c2)
                lvl_max = max(lvl_max, bv3_item<2, 2, LOCAL, CC, IT>(rowptr, col, node_off, hop_off, ord2[idx], cap2, (wq & 1) * 32 + lane,
                                                     bar_group + 1 + pr, gslice + (size_t)pr * half, out, ro, levels, overflow));
        } else {                                                     // up to 32 nodes: four graphs, a warp each
            const int64_t idx = 4 * (t - c_big - items2) + wq;
            if (idx < c3)
                lvl_max = max(lvl_max, bv3_item<1, 1, LOCAL, CC, IT>(rowptr, col, node_off, hop_off, ord3[idx], cap1, lane, 0,
                                                     gslice + (size_t)wq * quarter, out, ro, levels, overflow));
        }
        bv3_sync<BV3_GW>(bar_group);                                 // the slice is re-partitioned / refilled by the next item
    }
    if (max_level) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) lvl_max = max(lvl_max, __shfl_xor_sync(0xffffffffu, lvl_max, o));
        if (lane == 0 && lvl_max > 0) atomicMax(max_level, lvl_max);
    }
}

// ---- batched graphs of 129..GNAN_APSP_BATCHED_MAX_NODES nodes: one CTA per graph, bit-parallel over 128 sources at a time -------
// The v3 pull on a whole CTA: thread t owns vertices t and t + BL_THREADS and keeps, per vertex, the bits of the chunk's sources
// s0..s0+127 that reach it (BL_W words). Level L: new[v] = (OR_{u in out(v)} frontier[u]) & ~visited[v]; a new bit s means
// hop[v][s0+s] = L and popc(new[v]) adds to row v's level-L count. A thread owns rows v of hop and cnt: no atomics. One
// __syncthreads_or per level ends the level loop of a chunk. The CTA first writes its graph's 255 / 0 background (coalesced
// 16-byte stores), then scatters the reached bytes and adds each chunk's counts into the rows. Neighbours come from the CSR.
// rscale (1/count, gnan_level_rscale's 1.0f / (float)count) without cnt: the counts are summed in the rscale rows themselves (exact
// integers in fp32) and each owner thread inverts its rows once after the last chunk.
constexpr int BL_THREADS = 512;
constexpr int BL_VPT = GNAN_APSP_BATCHED_MAX_NODES / BL_THREADS;   // vertices per thread
constexpr int BL_W = 4;                                              // source words per vertex: 128 sources per chunk

__global__ void __launch_bounds__(BL_THREADS, 2)
apsp_batched_large_kernel(const int32_t *__restrict__ rowptr, const int32_t *__restrict__ col, const int32_t *__restrict__ node_off,
                          const int64_t *__restrict__ hop_off, int B, uint8_t *__restrict__ hop, int32_t *__restrict__ cnt,
                          float *__restrict__ rscale, int nbins, int32_t *__restrict__ overflow, int32_t *__restrict__ max_level,
                          const int32_t *__restrict__ order)
{
    __shared__ __align__(16) uint32_t fr[2][GNAN_APSP_BATCHED_MAX_NODES * BL_W];   // frontier rows [n][BL_W], by level parity
    const int tid = threadIdx.x;
    const int n_large = order[4 + 4 * (size_t)B];
    const int32_t *list = order + 5 + 4 * (size_t)B;
    int lvl_max = 0;
    for (int t = blockIdx.x; t < n_large; t += gridDim.x) {
        const int64_t b = list[t];
        const int n0 = node_off[b], n = node_off[b + 1] - n0;
        uint8_t *gb = hop + hop_off[b];
        int32_t *gc = cnt ? cnt + (int64_t)n0 * nbins : nullptr;
        float *gr = rscale ? rscale + (int64_t)n0 * nbins : nullptr;
        float *gf = gc ? nullptr : gr;                               // the count rows in fp32 when there is no int32 table
        // background: head bytes up to the first 16-byte boundary, vector body, tail bytes
        const int total = n * n;
        const int head = min(total, (int)((16 - (reinterpret_cast<uintptr_t>(gb) & 15)) & 15));
        if (tid < head) gb[tid] = GNAN_HOP_UNREACHABLE;
        const int body = (total - head) / 16;
        for (int i = tid; i < body; i += BL_THREADS)
            *reinterpret_cast<uint4 *>(gb + head + (size_t)i * 16) = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
        const int tail0 = head + body * 16;
        if (tid < 16 && tail0 + tid < total) gb[tail0 + tid] = GNAN_HOP_UNREACHABLE;
        if (gc)
            for (int i = tid; i < n * nbins; i += BL_THREADS) gc[i] = 0;
        if (gf)
            for (int i = tid; i < n * nbins; i += BL_THREADS) gf[i] = 0.f;
        __syncthreads();
        int reached[BL_VPT];
#pragma unroll
        for (int k = 0; k < BL_VPT; ++k) {
            const int v = tid + k * BL_THREADS;
            reached[k] = 1;
            if (v < n) {
                gb[(size_t)v * n + v] = 0;
                if (gc) gc[(int64_t)v * nbins] = 1;
                if (gf) gf[(int64_t)v * nbins] = 1.f;
            }
        }
        for (int s0 = 0; s0 < n; s0 += 32 * BL_W) {
            uint32_t vis[BL_VPT][BL_W];
#pragma unroll
            for (int k = 0; k < BL_VPT; ++k) {
                const int v = tid + k * BL_THREADS, rel = v - s0;
#pragma unroll
                for (int ww = 0; ww < BL_W; ++ww) vis[k][ww] = (rel >= 0 && (rel >> 5) == ww) ? 1u << (rel & 31) : 0u;
                if (v < n) bv3_store_row<BL_W>(fr[0] + v * BL_W, vis[k]);
            }
            __syncthreads();
            for (int level = 1; level <= n; ++level) {
                const uint32_t *fc = fr[(level - 1) & 1];
                uint32_t *fn = fr[level & 1];
                const uint8_t lv = (uint8_t)min(level, 254);
                bool any = false;
#pragma unroll
                for (int k = 0; k < BL_VPT; ++k) {
                    const int v = tid + k * BL_THREADS;
                    if (v < n) {
                        uint32_t acc[BL_W] = {0u, 0u, 0u, 0u};
                        const int e1 = rowptr[n0 + v + 1];
                        for (int e = rowptr[n0 + v]; e < e1; ++e) {          // neighbours outside the graph are ignored
                            const int u = __ldg(col + e) - n0;
                            if (u >= 0 && u < n) bv3_or_row<BL_W>(fc + u * BL_W, acc);
                        }
                        int newc = 0;
#pragma unroll
                        for (int ww = 0; ww < BL_W; ++ww) {
                            acc[ww] &= ~vis[k][ww];
                            vis[k][ww] |= acc[ww];
                            newc += __popc(acc[ww]);
                        }
                        bv3_store_row<BL_W>(fn + v * BL_W, acc);
                        if (newc) {
                            any = true;
                            uint8_t *rowp = gb + (size_t)v * n + s0;
#pragma unroll
                            for (int ww = 0; ww < BL_W; ++ww) {
                                uint32_t m = acc[ww];
                                while (m) {
                                    rowp[ww * 32 + __ffs(m) - 1] = lv;
                                    m &= m - 1;
                                }
                            }
                            if (level > 254 || level >= nbins - 1) atomicExch(overflow, 1);
                            else if (gc) gc[(int64_t)v * nbins + level] += newc;
                            else if (gf) gf[(int64_t)v * nbins + level] += (float)newc;
                            reached[k] += newc;
                        }
                    }
                }
                if (!__syncthreads_or(any)) break;
                lvl_max = max(lvl_max, level);
            }
        }
#pragma unroll
        for (int k = 0; k < BL_VPT; ++k) {
            const int v = tid + k * BL_THREADS;
            if (v >= n) continue;
            if (gc) gc[(int64_t)v * nbins + nbins - 1] = n - reached[k];
            if (gf) gf[(int64_t)v * nbins + nbins - 1] = (float)(n - reached[k]);
            if (gr)
                for (int d = 0; d < nbins; ++d) {                   // as level_rscale_kernel
                    const float c = gc ? (float)gc[(int64_t)v * nbins + d] : gr[(int64_t)v * nbins + d];
                    gr[(int64_t)v * nbins + d] = c > 0.f ? 1.0f / c : 0.f;
                }
        }
    }
    if (max_level && tid == 0 && lvl_max > 0) atomicMax(max_level, lvl_max);   // lvl_max is uniform over the CTA
}

// ---- the fused BFS + graph readout on graphs of 129..GNAN_APSP_BATCHED_MAX_NODES nodes: one CTA per graph -------------------
// The sources advance 128 at a time as in apsp_batched_large_kernel, but the pull runs over IN-neighbours: vertex v keeps the bits
// of the chunk's sources s that reach it, and a new bit (v, s) at level L means d(s -> v) = L, i.e. hop[s][v] = L. So v is column
// j = v of the readout and the level size count(s, L) = cnt[s][L] of row s is a column count over the CTA's vertices: every new
// bit adds 1 to the chunk's shared-memory integer counter of its source, and the counters are complete when the level's barrier
// has passed. Each vertex then adds P[v,L] = sum over its new sources (ascending) of 1/count(s,L) and folds it at once, as the v3
// readout does: colw[v,:] += T[L,:] p in registers, Q[L,:] += S[v,:] p as one warp sum into the warp's own [nbins][C] slot (added
// to across chunks; the slots are added in warp order at the end). colw sums one term per (chunk, level), up to 8 x 63 for a graph
// of 1024 nodes, and the unreachable bin one term per source that does not reach v, up to 1023: both are accumulated in fp64 (in
// fp32, 1024-node graphs missed the 1e-5 * A bound of the float64 reference). Exact on directed graphs in one pass, no symmetry test. The
// unreachable bin: after each chunk, 1/(n - reached_s) over the chunk's sources that did not reach v, in a register until the end.
// Level 0 contributes 1 to every vertex once. The in-neighbour bit matrix [n][ceil(n/32)] is built in shared memory from the
// graph's own edge segment (atomicOr: duplicates and endpoints beyond the graph set the status bits, as the v3 kernels); up to 4
// in-neighbours of a vertex are cached as 16-bit halves of two registers, longer rows walk their bit row. Nothing but out, colw,
// Q and the status words reaches global memory. Dynamic shared memory and the block size follow the batch's largest graph.
constexpr int BRL_MAX_THREADS = 512;
constexpr int BRL_VPT = GNAN_APSP_BATCHED_MAX_NODES / BRL_MAX_THREADS;   // vertices per thread
constexpr int BRL_SRC = 32 * BL_W;                                       // sources per chunk

// threads per CTA: one per vertex up to 512 nodes (a batch holds few large graphs, so each one's latency is what counts), two above;
// at least one per source of a chunk
inline int brl_threads(int cap) { return std::min(BRL_MAX_THREADS, std::max(BRL_SRC, (cap + 31) / 32 * 32)); }
// frontier rows [2][cap][BL_W], in-neighbour bits [cap][ceil(cap/32)], per-warp Q [NW][nbins][CC] + out [NW][CC], source counters
// [3][BRL_SRC] (by level mod 3: filled at L, read after the barrier of L, zeroed at L + 2), 1/(n - reached) [BRL_SRC]
inline size_t brl_need(int cap, int nthreads, int nbins, int CC)
{
    return (size_t)2 * cap * BL_W * 4 + (size_t)cap * ((cap + 31) / 32) * 4 + (size_t)(nthreads / 32) * (nbins + 1) * CC * 4 +
           (size_t)4 * BRL_SRC * 4;
}

// the vertex share of bin d: colw += T[d,:] p, the warp's Q slot [d,:] += the warp sum of S[v,:] p (all threads call it)
template <int CC, typename PT>
__device__ __forceinline__ void brl_fold(int d, const PT (&p)[BRL_VPT], const float (&s)[BRL_VPT][CC], double (&cw)[BRL_VPT][CC],
                                         float *sqw, const Bv3Readout &r, int lane)
{
#pragma unroll
    for (int c = 0; c < CC; ++c) {
        if (c < r.Cr) {
            const double t = __ldg(r.T + d * r.Cr + c);
#pragma unroll
            for (int k = 0; k < BRL_VPT; ++k) cw[k][c] = fma(t, (double)p[k], cw[k][c]);
        }
        if (c < r.C) {
            float q = s[0][c] * (float)p[0];
#pragma unroll
            for (int k = 1; k < BRL_VPT; ++k) q = fmaf(s[k][c], (float)p[k], q);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
            if (lane == 0) sqw[d * CC + c] += q;
        }
    }
}

template <typename IT, int CC>
__global__ void __launch_bounds__(BRL_MAX_THREADS, CC > 1 ? 1 : 2)
bfs_readout_large_kernel(const IT *__restrict__ src, const IT *__restrict__ dst, const int32_t *__restrict__ edge_off,
                         const int32_t *__restrict__ node_off, int B, int cap, int nbins, Bv3Readout r, int32_t *__restrict__ status,
                         int32_t *__restrict__ overflow, int32_t *__restrict__ max_level, const int32_t *__restrict__ order)
{
    extern __shared__ __align__(16) uint8_t smL[];
    const int tid = threadIdx.x, NT = blockDim.x, lane = tid & 31, warp = tid >> 5, NW = NT >> 5, nq = nbins * CC;
    uint32_t *fr = reinterpret_cast<uint32_t *>(smL);                     // [2][cap][BL_W]
    uint32_t *adj = fr + 2 * cap * BL_W;                                   // [n][AW] of [cap][ceil(cap/32)]
    float *sq = reinterpret_cast<float *>(adj + cap * ((cap + 31) / 32));  // [NW][nbins][CC]
    float *so = sq + NW * nq;                                              // [NW][CC]
    int *cnt = reinterpret_cast<int *>(so + NW * CC);                      // [3][BRL_SRC]
    float *urc = reinterpret_cast<float *>(cnt + 3 * BRL_SRC);             // [BRL_SRC]
    float *sqw = sq + warp * nq;
    const int n_large = order[4 + 4 * (size_t)B];
    const int32_t *list = order + 5 + 4 * (size_t)B;
    int lvl_max = 0;
    for (int t = blockIdx.x; t < n_large; t += gridDim.x) {
        const int64_t b = list[t];
        const int n0 = node_off[b], n = node_off[b + 1] - n0, AW = (n + 31) / 32;
        for (int i = tid; i < n * AW; i += NT) adj[i] = 0u;
        for (int i = tid; i < NW * (nq + CC); i += NT) sq[i] = 0.f;
        __syncthreads();
        const int e0 = edge_off[b], e1 = edge_off[b + 1];
        int flags = 0;
        for (int e = e0 + tid; e < e1; e += NT) {                          // edge s -> d: bit s of d's in-neighbour row
            const uint32_t s = local_index(src[e]), d = local_index(dst[e]);
            if (s < (uint32_t)n && d < (uint32_t)n) {
                const uint32_t bit = 1u << (s & 31);
                if (atomicOr(adj + d * AW + (s >> 5), bit) & bit) flags |= 2;
            } else {
                flags |= 1;
            }
        }
        if (flags) atomicOr(status, flags);
        __syncthreads();

        float s[BRL_VPT][CC], p[BRL_VPT];
        double cw[BRL_VPT][CC], U[BRL_VPT];
        uint32_t nb[BRL_VPT][2];
        int dg[BRL_VPT];                                                   // in-degree; > 4: walk the bit row
#pragma unroll
        for (int k = 0; k < BRL_VPT; ++k) {
            const int v = tid + k * NT;
            const bool mine = v < n;
#pragma unroll
            for (int c = 0; c < CC; ++c) {
                s[k][c] = (mine && c < r.C) ? r.S[(int64_t)(n0 + v) * r.C + c] : 0.f;
                cw[k][c] = 0.0;
            }
            U[k] = 0.0;
            p[k] = mine ? 1.f : 0.f;                                       // level 0: v itself, count 1
            nb[k][0] = nb[k][1] = 0u;
            dg[k] = 0;
            if (mine) {
                const uint32_t *arow = adj + v * AW;
                for (int ww = 0; ww < AW; ++ww) dg[k] += __popc(arow[ww]);
                if (dg[k] <= 4) {
                    int j = 0;
                    for (int ww = 0; ww < AW; ++ww)
                        for (uint32_t m = arow[ww]; m; m &= m - 1, ++j) {
                            const uint32_t u = (uint32_t)(ww * 32 + __ffs(m) - 1) << (16 * (j & 1));
                            if (j < 2) nb[k][0] |= u;
                            else nb[k][1] |= u;
                        }
                }
            }
        }
        brl_fold<CC>(0, p, s, cw, sqw, r, lane);
        for (int s0 = 0; s0 < n; s0 += BRL_SRC) {
            uint32_t vis[BRL_VPT][BL_W];
#pragma unroll
            for (int k = 0; k < BRL_VPT; ++k) {
                const int v = tid + k * NT, rel = v - s0;
#pragma unroll
                for (int ww = 0; ww < BL_W; ++ww) vis[k][ww] = (rel >= 0 && (rel >> 5) == ww) ? 1u << (rel & 31) : 0u;
                if (v < n) bv3_store_row<BL_W>(fr + v * BL_W, vis[k]);
            }
            for (int i = tid; i < 3 * BRL_SRC; i += NT) cnt[i] = 0;
            int reach = 1;                                                 // thread tid < BRL_SRC: vertices reached by source s0 + tid
            __syncthreads();
            for (int level = 1; level <= n; ++level) {
                const uint32_t *fc = fr + ((level - 1) & 1) * cap * BL_W;
                uint32_t *fn = fr + (level & 1) * cap * BL_W;
                int *cl = cnt + (level % 3) * BRL_SRC;
                if (tid < BRL_SRC) cnt[((level + 1) % 3) * BRL_SRC + tid] = 0;
                bool any = false;
#pragma unroll
                for (int k = 0; k < BRL_VPT; ++k) {
                    const int v = tid + k * NT;
                    if (v >= n) continue;
                    uint32_t acc[BL_W] = {0u, 0u, 0u, 0u};
                    if (dg[k] <= 4) {
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            if (j < dg[k]) bv3_or_row<BL_W>(fc + ((nb[k][j >> 1] >> (16 * (j & 1))) & 0xffffu) * BL_W, acc);
                    } else {
                        const uint32_t *arow = adj + v * AW;
                        for (int ww = 0; ww < AW; ++ww)
                            for (uint32_t m = arow[ww]; m; m &= m - 1) bv3_or_row<BL_W>(fc + (ww * 32 + __ffs(m) - 1) * BL_W, acc);
                    }
                    bool nw = false;
#pragma unroll
                    for (int ww = 0; ww < BL_W; ++ww) {
                        acc[ww] &= ~vis[k][ww];
                        vis[k][ww] |= acc[ww];
                        nw |= acc[ww] != 0u;
                        for (uint32_t m = acc[ww]; m; m &= m - 1) atomicAdd(cl + ww * 32 + __ffs(m) - 1, 1);
                    }
                    bv3_store_row<BL_W>(fn + v * BL_W, acc);
                    if (nw) {
                        any = true;
                        if (level >= nbins - 1) atomicExch(overflow, 1);
                    }
                }
                if (!__syncthreads_or(any)) break;
                lvl_max = max(lvl_max, level);
                if (tid < BRL_SRC) reach += cl[tid];
                if (level < nbins - 1) {                                   // P[v, level] over v's new sources, from its frontier row
#pragma unroll
                    for (int k = 0; k < BRL_VPT; ++k) {
                        const int v = tid + k * NT;
                        p[k] = 0.f;
                        if (v >= n) continue;
                        const uint4 q = *reinterpret_cast<const uint4 *>(fn + v * BL_W);
                        const uint32_t w4[BL_W] = {q.x, q.y, q.z, q.w};
#pragma unroll
                        for (int ww = 0; ww < BL_W; ++ww)
                            for (uint32_t m = w4[ww]; m; m &= m - 1) p[k] += __frcp_rn((float)cl[ww * 32 + __ffs(m) - 1]);
                    }
                    brl_fold<CC>(level, p, s, cw, sqw, r, lane);
                }
            }
            if (tid < BRL_SRC) urc[tid] = (s0 + tid < n && reach < n) ? __frcp_rn((float)(n - reach)) : 0.f;
            __syncthreads();
            const int nsrc = min(BRL_SRC, n - s0);
#pragma unroll
            for (int k = 0; k < BRL_VPT; ++k) {
                if (tid + k * NT >= n) continue;
#pragma unroll
                for (int ww = 0; ww < BL_W; ++ww) {
                    const int left = nsrc - ww * 32;
                    for (uint32_t m = ~vis[k][ww] & (left >= 32 ? 0xffffffffu : (left > 0 ? (1u << left) - 1u : 0u)); m; m &= m - 1)
                        U[k] += urc[ww * 32 + __ffs(m) - 1];
                }
            }
            __syncthreads();                                               // the next chunk rewrites fr, cnt and urc
        }
        brl_fold<CC>(nbins - 1, U, s, cw, sqw, r, lane);
#pragma unroll
        for (int k = 0; k < BRL_VPT; ++k) {
            const int v = tid + k * NT;
            if (v < n) {
#pragma unroll
                for (int c = 0; c < CC; ++c)
                    if (c < r.Cr) r.colw[(int64_t)(n0 + v) * r.Cr + c] = (float)cw[k][c];
            }
        }
        // out[b,c] = sum_v S[v,c] colw[v,c']: a warp sum each, then the warps in order
#pragma unroll
        for (int c = 0; c < CC; ++c) {
            if (c < r.C) {
                const int cc = r.Cr == 1 ? 0 : c;
                float q = s[0][c] * (float)cw[0][cc];
#pragma unroll
                for (int k = 1; k < BRL_VPT; ++k) q = fmaf(s[k][c], (float)cw[k][cc], q);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
                if (lane == 0) so[warp * CC + c] = q;
            }
        }
        __syncthreads();
        for (int i = tid; i < nbins * r.C; i += NT) {                      // Q[b] in full (empty bins: 0), coalesced
            const int d = i / r.C, c = i - d * r.C;
            float q = 0.f;
            for (int w = 0; w < NW; ++w) q += sq[w * nq + d * CC + c];
            r.Q[(int64_t)b * nbins * r.C + i] = q;
        }
        if (tid < r.C) {
            float q = 0.f;
            for (int w = 0; w < NW; ++w) q += so[w * CC + tid];
            r.out[b * r.C + tid] = q;
        }
        __syncthreads();                                                   // the next graph rewrites the shared memory
    }
    if (max_level && tid == 0 && lvl_max > 0) atomicMax(max_level, lvl_max);   // lvl_max is uniform over the CTA
}

// ---- one large graph: one warp per source, queue + bitmap in the workspace -----------------------------------------
__global__ void __launch_bounds__(256)
apsp_bfs_kernel(const int32_t *__restrict__ rowptr, const int32_t *__restrict__ col, int N, int src_begin, int src_end,
                uint8_t *__restrict__ hop, int64_t ld, int32_t *__restrict__ cnt, int nbins, int32_t *__restrict__ overflow,
                int32_t *__restrict__ queues, uint32_t *__restrict__ bitmaps, int bm_words, int64_t nwarps)
{
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (warp >= nwarps) return;  // queues / bitmaps are sized for nwarps warps
    int32_t *q = queues + warp * (int64_t)N;
    uint32_t *bm = bitmaps + warp * (int64_t)bm_words;
    for (int64_t s = src_begin + warp; s < src_end; s += nwarps) {
        uint8_t *row = hop + (s - src_begin) * ld;
        for (int64_t v = lane * 16; v < ld; v += 512)
            *reinterpret_cast<uint4 *>(row + v) = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
        for (int t = lane; t < bm_words; t += 32) bm[t] = 0u;
        int32_t *crow = cnt ? cnt + (s - src_begin) * nbins : nullptr;
        if (crow)
            for (int d = lane; d < nbins; d += 32) crow[d] = 0;
        __syncwarp();
        if (lane == 0) {
            q[0] = (int32_t)s;
            bm[s >> 5] = 1u << (s & 31);
            row[s] = 0;
            if (crow) crow[0] = 1;
        }
        __syncwarp();
        int head = 0, tail = 1, level = 0;
        while (head < tail) {
            ++level;
            const uint8_t lv = (uint8_t)min(level, 254);
            int new_tail = tail;
            for (int base = head; base < tail; base += 32) {
                const int idx = base + lane;
                int e0 = 0, e1 = 0;
                if (idx < tail) {
                    const int v = q[idx];
                    e0 = rowptr[v];
                    e1 = rowptr[v + 1];
                }
                // lanes walk their own adjacency lists; claims go through the warp-private bitmap
                int maxdeg = e1 - e0;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) maxdeg = max(maxdeg, __shfl_xor_sync(0xffffffffu, maxdeg, o));
                for (int k = 0; k < maxdeg; ++k) {
                    bool won = false;
                    int t = -1;
                    if (e0 + k < e1) {
                        t = col[e0 + k];
                        const uint32_t bit = 1u << (t & 31);
                        const uint32_t old = atomicOr(bm + (t >> 5), bit);
                        won = !(old & bit);
                    }
                    const uint32_t mask = __ballot_sync(0xffffffffu, won);
                    if (won) {
                        q[new_tail + __popc(mask & ((1u << lane) - 1))] = t;
                        row[t] = lv;
                    }
                    new_tail += __popc(mask);
                }
            }
            __syncwarp();
            const int newc = new_tail - tail;
            if (newc > 0) {
                if (lane == 0) {
                    if (level > 254 || level >= nbins - 1) atomicExch(overflow, 1);
                    else if (crow) crow[level] = newc;
                }
            }
            head = tail;
            tail = new_tail;
        }
        if (lane == 0 && crow) crow[nbins - 1] = N - tail;
        __syncwarp();
    }
}


// ---- one large graph, bit-parallel multi-source BFS ---------------------------------------------------------------------
constexpr int MSBFS_FLAG_STRIDE = 32;            // int32 per level flag: one 128-byte line each
// A batch of SB = 32*W sources (= hop-matrix COLUMNS s0..s0+SB) is advanced together: every vertex v keeps W words of
// "reached-from" bits. Level L is a PULL over v's out-neighbours u (edge v -> u): v reaches source s in L steps iff some u
// reaches s in L-1 steps, so the value produced for (v, s) is dist(v -> s) = hop[v][s] and each vertex writes its OWN row
// segment hop[v][s0 .. s0+SB) (contiguous bytes; no transposed CSR, no transpose pass, directed graphs included).
// One launch per level; `changed` tells the host-side loop when the batch has converged.
__global__ void msbfs_init_kernel(int N, int s0, int SB, int W, uint32_t *__restrict__ visited, uint32_t *__restrict__ frontier,
                                  int row_begin, int row_end, uint8_t *__restrict__ hop, int64_t ld, int32_t *__restrict__ cnt, int nbins)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)N * W) return;
    const int v = (int)(t / W), w = (int)(t % W);
    uint32_t bits = 0u;
    const int rel = v - s0 - w * 32;                     // v itself is source number w*32 + rel of the batch
    if (rel >= 0 && rel < 32 && w * 32 + rel < SB) bits = 1u << rel;
    visited[t] = bits;
    frontier[t] = bits;
    if (v >= row_begin && v < row_end) {
        uint8_t *seg = hop + (int64_t)(v - row_begin) * ld + s0 + w * 32;
        const int nvalid = min(32, SB - w * 32);
        if (nvalid == 32 && bits == 0u) {                // ld % 16 == 0 and s0 % 32 == 0: 16-byte aligned
            const uint4 ff = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
            reinterpret_cast<uint4 *>(seg)[0] = ff;
            reinterpret_cast<uint4 *>(seg)[1] = ff;
        } else {
            for (int b = 0; b < nvalid; ++b) seg[b] = (bits >> b) & 1u ? 0 : GNAN_HOP_UNREACHABLE;
        }
        if (s0 == 0 && w == 0)                           // row padding columns [N, ld)
            for (int64_t c = N; c < ld; ++c) hop[(int64_t)(v - row_begin) * ld + c] = GNAN_HOP_UNREACHABLE;
        if (bits && cnt) atomicAdd(cnt + (int64_t)(v - row_begin) * nbins, 1);
    }
}

__global__ void msbfs_level_kernel(const int32_t *__restrict__ rowptr, const int32_t *__restrict__ col, int N, int s0, int W,
                                   int level, uint32_t *__restrict__ visited, const uint32_t *__restrict__ frontier,
                                   uint32_t *__restrict__ next, int row_begin, int row_end, uint8_t *__restrict__ hop, int64_t ld,
                                   int32_t *__restrict__ cnt, int nbins, int32_t *__restrict__ changed, int32_t *__restrict__ overflow)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    // the batch converged at an earlier level: nothing left to do. One flag per 128-byte line: the flag of THIS level is
    // being stored to by other CTAs while the previous one is read (sharing a line cost 2x on the whole BFS).
    if (level > 1 && changed[(level - 1) * MSBFS_FLAG_STRIDE] == 0) return;
    const bool valid = t < (int64_t)N * W;
    const int v = valid ? (int)(t / W) : 0, w = (int)(t % W);
    uint32_t vis = 0xffffffffu, acc = 0u;
    if (valid) {
        vis = visited[t];
        if (vis != 0xffffffffu) {
            const int e1 = rowptr[v + 1];
            for (int e = rowptr[v]; e < e1; ++e) acc |= frontier[(int64_t)col[e] * W + w];
        }
    }
    const uint32_t nw = acc & ~vis;
    if (valid) next[t] = nw;
    if (__any_sync(0xffffffffu, nw != 0u) && (threadIdx.x & 31) == 0) changed[level * MSBFS_FLAG_STRIDE] = 1;
    if (nw) {
        visited[t] = vis | nw;
        if (level > 254 || level >= nbins - 1) *overflow = 1;
        if (v >= row_begin && v < row_end) {
            uint8_t *seg = hop + (int64_t)(v - row_begin) * ld + s0 + w * 32;
            uint32_t m = nw;
            const uint8_t lv = (uint8_t)min(level, 254);
            while (m) {
                seg[__ffs(m) - 1] = lv;
                m &= m - 1;
            }
            if (cnt && level < nbins - 1) atomicAdd(cnt + (int64_t)(v - row_begin) * nbins + level, __popc(nw));
        }
    }
}

// cnt[v][nbins-1] = (#columns) - sum of the finite levels
__global__ void msbfs_unreachable_kernel(int rows, int ncols, int32_t *__restrict__ cnt, int nbins)
{
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= rows) return;
    int s = 0;
    for (int d = 0; d < nbins - 1; ++d) s += cnt[(int64_t)v * nbins + d];
    cnt[(int64_t)v * nbins + nbins - 1] = ncols - s;
}

// ---- converters ------------------------------------------------------------------------------------------------------
__global__ void hops_to_reference_kernel(const uint8_t *__restrict__ hop, int64_t R, int64_t N, int64_t ld,
                                         const int32_t *__restrict__ cnt, int nbins, float *__restrict__ nd, float *__restrict__ nm)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= R * N) return;
    const int64_t i = t / N, j = t % N;
    const int h = hop[i * ld + j];
    if (nd) nd[t] = h == GNAN_HOP_UNREACHABLE ? 0.f : 1.0f / ((float)h + 1.0f);
    if (nm) nm[t] = (float)cnt[i * nbins + min(h, nbins - 1)];
}

__global__ void hops_from_reference_kernel(const float *__restrict__ nd, const float *__restrict__ nm, int64_t R, int64_t N,
                                           uint8_t *__restrict__ hop, int64_t ld, int32_t *__restrict__ cnt, int nbins,
                                           int32_t *__restrict__ overflow)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= R * ld) return;
    const int64_t i = t / ld, j = t % ld;
    if (j >= N) { hop[t] = GNAN_HOP_UNREACHABLE; return; }
    const float v = nd[i * N + j];
    int h = GNAN_HOP_UNREACHABLE;
    if (v > 0.f) {
        const float hf = rintf(1.0f / v - 1.0f);
        if (hf > 254.f || hf >= (float)(nbins - 1)) { atomicExch(overflow, 1); h = 254; }
        else h = (int)hf;
    }
    hop[t] = (uint8_t)h;
    if (cnt) {
        const int b = min(h, nbins - 1);
        if (nm) cnt[i * nbins + b] = (int32_t)rintf(nm[i * N + j]);   // every writer of a bin stores the same value
        else atomicAdd(cnt + i * nbins + b, 1);
    }
}

}  // namespace

extern "C" size_t gnan_apsp_bfs_workspace_bytes(int32_t N, int32_t n_sources)
{
    if (N <= 0 || n_sources <= 0) return 0;
    const int64_t nwarps = std::min<int64_t>(n_sources, (int64_t)gnan_sm_count() * 8);
    const int64_t bm_words = (N + 31) / 32;
    return (size_t)nwarps * ((size_t)N * 4 + (size_t)bm_words * 4);
}

extern "C" int gnan_apsp_bfs(const int32_t *rowptr, const int32_t *col, int32_t N, int32_t src_begin, int32_t src_end,
                             uint8_t *hop, int64_t ld_hop, int32_t *cnt, int32_t nbins, int32_t *overflow_flag,
                             void *workspace, size_t workspace_bytes, gnan_stream_t stream)
{
    GNAN_REQUIRE(N >= 0 && src_begin >= 0 && src_end >= src_begin && src_end <= N, "apsp_bfs: bad source range [%d,%d) N=%d", src_begin, src_end, N);
    const int ns = src_end - src_begin;
    if (ns == 0) return GNAN_OK;
    GNAN_REQUIRE(rowptr && hop && overflow_flag, "apsp_bfs: NULL pointer");
    GNAN_REQUIRE(ld_hop >= N && ld_hop % 16 == 0 && ((uintptr_t)hop % 16) == 0, "apsp_bfs: hop rows must be 16-byte aligned, ld %% 16 == 0");
    GNAN_REQUIRE(!cnt || (nbins >= 2 && nbins <= 256), "apsp_bfs: nbins %d out of [2,256]", nbins);
    const size_t need = gnan_apsp_bfs_workspace_bytes(N, ns);
    if (!workspace || workspace_bytes < need) {
        gnan_set_error("apsp_bfs: workspace %zu < %zu bytes", workspace_bytes, need);
        return GNAN_ERR_WORKSPACE;
    }
    const int64_t nwarps = std::min<int64_t>(ns, (int64_t)gnan_sm_count() * 8);
    const int bm_words = (N + 31) / 32;
    int32_t *queues = (int32_t *)workspace;
    uint32_t *bitmaps = (uint32_t *)(queues + nwarps * (int64_t)N);
    const int blocks = (int)ceil_div64(nwarps, 8);
    apsp_bfs_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(rowptr, col, N, src_begin, src_end, hop, ld_hop, cnt,
                                                               cnt ? nbins : 256, overflow_flag, queues, bitmaps, bm_words, nwarps);
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}


// ---- bit-parallel multi-source BFS (large graphs) ------------------------------------------------------------------------
constexpr int MSBFS_W = 32;                      // 1024 sources per batch
constexpr int MSBFS_MAX_LEVELS = 272;            // per-level "anything new?" flags (levels past 254 only raise overflow)
constexpr int MSBFS_GROUP = 8;                   // levels launched per host round trip

extern "C" size_t gnan_apsp_msbfs_workspace_bytes(int32_t N)
{
    return N > 0 ? 3 * sizeof(uint32_t) * (size_t)N * MSBFS_W + sizeof(int32_t) * MSBFS_MAX_LEVELS * MSBFS_FLAG_STRIDE : 0;
}

// Rows [row_begin,row_end) of the hop matrix of an N-node graph (all N columns). Unlike every other entry point this one
// SYNCHRONISES the stream: the number of BFS levels is data dependent and is read back once per level group.
extern "C" int gnan_apsp_msbfs(const int32_t *rowptr, const int32_t *col, int32_t N, int32_t row_begin, int32_t row_end,
                               uint8_t *hop, int64_t ld_hop, int32_t *cnt, int32_t nbins, int32_t *overflow_flag,
                               void *workspace, size_t workspace_bytes, gnan_stream_t stream)
{
    GNAN_REQUIRE(N >= 0 && row_begin >= 0 && row_end >= row_begin && row_end <= N, "apsp_msbfs: bad row range [%d,%d) N=%d", row_begin, row_end, N);
    if (row_end == row_begin || N == 0) return GNAN_OK;
    GNAN_REQUIRE(rowptr && hop && overflow_flag, "apsp_msbfs: NULL pointer");
    GNAN_REQUIRE(ld_hop >= N && ld_hop % 16 == 0, "apsp_msbfs: ld_hop must be >= N and a multiple of 16");
    GNAN_REQUIRE(!cnt || (nbins >= 2 && nbins <= 256), "apsp_msbfs: nbins %d out of [2,256]", nbins);
    const size_t need = gnan_apsp_msbfs_workspace_bytes(N);
    if (!workspace || workspace_bytes < need) {
        gnan_set_error("apsp_msbfs: workspace %zu < %zu bytes", workspace_bytes, need);
        return GNAN_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int rows = row_end - row_begin;
    const int nb = cnt ? nbins : 256;
    uint32_t *visited = (uint32_t *)workspace;
    uint32_t *bufA = visited + (size_t)N * MSBFS_W, *bufB = bufA + (size_t)N * MSBFS_W;
    int32_t *changed = (int32_t *)(bufB + (size_t)N * MSBFS_W);
    if (cnt) GNAN_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int32_t) * (size_t)rows * nb, st));
    const unsigned blocks = (unsigned)ceil_div64((int64_t)N * MSBFS_W, 256);
    for (int s0 = 0; s0 < N; s0 += 32 * MSBFS_W) {
        const int SB = std::min(32 * MSBFS_W, N - s0);
        uint32_t *frontier = bufA, *next = bufB;
        msbfs_init_kernel<<<blocks, 256, 0, st>>>(N, s0, SB, MSBFS_W, visited, frontier, row_begin, row_end, hop, ld_hop, cnt, nb);
        GNAN_LAUNCH_OK();
        GNAN_CUDA(cudaMemsetAsync(changed, 0, sizeof(int32_t) * MSBFS_MAX_LEVELS * MSBFS_FLAG_STRIDE, st));
        int level = 0;
        for (;;) {
            for (int k = 0; k < MSBFS_GROUP; ++k) {          // levels after convergence return at once (changed[level-1] == 0)
                ++level;
                msbfs_level_kernel<<<blocks, 256, 0, st>>>(rowptr, col, N, s0, MSBFS_W, level, visited, frontier, next, row_begin,
                                                           row_end, hop, ld_hop, cnt, nb, changed, overflow_flag);
                GNAN_LAUNCH_OK();
                std::swap(frontier, next);
            }
            int32_t h = 0;
            GNAN_CUDA(cudaMemcpyAsync(&h, changed + level * MSBFS_FLAG_STRIDE, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
            GNAN_CUDA(cudaStreamSynchronize(st));
            if (!h || level + MSBFS_GROUP >= MSBFS_MAX_LEVELS) break;
        }
    }
    if (cnt) {
        msbfs_unreachable_kernel<<<(unsigned)ceil_div64(rows, 256), 256, 0, st>>>(rows, N, cnt, nb);
        GNAN_LAUNCH_OK();
    }
    return GNAN_OK;
}

// bv3_classify_kernel into order_ws ([4*B+4] words, [5*B+5] when max_n > 128)
static int classify_by_size(const int32_t *node_off, int32_t B, int32_t max_n, int32_t *order_ws, cudaStream_t st)
{
    GNAN_CUDA(cudaMemsetAsync(order_ws, 0, 4 * sizeof(int32_t), st));
    if (max_n > 32 * BV3_MAX_W) GNAN_CUDA(cudaMemsetAsync(order_ws + 4 * (size_t)B + 4, 0, sizeof(int32_t), st));
    bv3_classify_kernel<<<(unsigned)ceil_div64(B, 256), 256, 0, st>>>(node_off, B, order_ws);
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}

// v3 launch on classes 0..3 of order_ws: groups of 4 warps; the group's slice holds one graph of 65..128 nodes, two of 33..64 or
// four of up to 32. max_n (at most 128) sizes the slices.
// CC > 0: the BFS fused with the graph readout (bv3_readout_run; ro holds its tensors, hop / cnt / rscale are NULL)
template <bool LOCAL, int CC = 0, typename IT = uint8_t>
static int launch_bv3(const int32_t *rowptr, const int32_t *col, const int32_t *node_off, const int64_t *hop_off, int32_t B, int32_t max_n,
                      uint8_t *hop, int32_t *cnt, float *rscale, int nb, bool levels, int32_t *overflow_flag, int32_t *max_level,
                      const int32_t *order_ws, Bv3EdgesT<IT> le, cudaStream_t st, Bv3Readout ro = Bv3Readout{})
{
    const int Wmax = (max_n + 31) / 32;
    auto need = [&](int cap, int W, int G) {
        return CC > 0 ? bv3_ro_need(cap, W, G, nb, CC) : bv3_need(cap, W, nb, levels, LOCAL);
    };
    size_t slice = 4 * need(std::min(max_n, 32), 1, 1);
    if (Wmax >= 2) slice = std::max(slice, 2 * need(std::min(max_n, 64), 2, 2));
    if (Wmax >= 3) slice = std::max(slice, need(max_n, Wmax, 4));
    const int gpc = (int)std::min<size_t>(bv3_max_groups(CC), (112 * 1024) / slice);     // two CTAs per SM
    if (gpc < 1) return GNAN_ERR_UNSUPPORTED;
    const size_t smem3 = slice * gpc;
    auto kernel = apsp_batched_v3_kernel<LOCAL, CC, IT>;
    static thread_local size_t cached_smem3 = 0;
    static thread_local int cached_gpc = 0, cached_per_sm3 = 0;
    if (cached_smem3 != smem3 || cached_gpc != gpc || cached_per_sm3 == 0) {
        GNAN_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem3));
        GNAN_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&cached_per_sm3, kernel, 32 * BV3_GW * gpc, smem3));
        cached_smem3 = smem3; cached_gpc = gpc;
    }
    const int blocks3 = (int)std::min<int64_t>(ceil_div64(B, gpc), (int64_t)std::max(cached_per_sm3, 1) * gnan_sm_count());
    kernel<<<blocks3, 32 * BV3_GW * gpc, smem3, st>>>(rowptr, col, node_off, hop_off, B, max_n, gpc, (int)slice, hop, cnt, rscale, nb,
                                                      overflow_flag, max_level, order_ws, le, ro);
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}

// graphs of more than 128 nodes in the batch: class 4 of bv3_classify_kernel (the caller has run it into order_ws [5*B+5]).
// B bounds the number of such graphs; CTAs past the end of the class exit at once.
static int launch_batched_large(const int32_t *rowptr, const int32_t *col, const int32_t *node_off, const int64_t *hop_off, int32_t B,
                                uint8_t *hop, int32_t *cnt, float *rscale, int nb, int32_t *overflow_flag, int32_t *max_level,
                                const int32_t *order_ws, cudaStream_t st)
{
    static thread_local int per_sm = 0;
    if (per_sm == 0) GNAN_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, apsp_batched_large_kernel, BL_THREADS, 0));
    const int blocks = (int)std::min<int64_t>(B, (int64_t)std::max(per_sm, 1) * gnan_sm_count());
    apsp_batched_large_kernel<<<blocks, BL_THREADS, 0, st>>>(rowptr, col, node_off, hop_off, B, hop, cnt, rscale, nb, overflow_flag,
                                                             max_level, order_ws);
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}

// graphs of at most 128 nodes: v3; graphs of 129..GNAN_APSP_BATCHED_MAX_NODES nodes: apsp_batched_large_kernel, one CTA each.
// rscale (optional): 1/count per (node, level) as fp32, what gnan_level_rscale would compute from cnt; cnt may then be NULL
extern "C" int gnan_apsp_bfs_batched_ex(const int32_t *rowptr, const int32_t *col, const int32_t *node_off, const int64_t *hop_off,
                                        int32_t B, int32_t max_n, uint8_t *hop, int32_t *cnt, float *rscale, int32_t nbins,
                                        int32_t *overflow_flag, int32_t *max_level, int32_t *order_ws, gnan_stream_t stream)
{
    GNAN_REQUIRE(B >= 0, "apsp_bfs_batched: negative batch");
    if (B == 0) return GNAN_OK;
    GNAN_REQUIRE(rowptr && node_off && hop_off && hop && overflow_flag, "apsp_bfs_batched: NULL pointer");
    GNAN_REQUIRE(order_ws, "apsp_bfs_batched: NULL order_ws");
    GNAN_REQUIRE(!(cnt || rscale) || (nbins >= 2 && nbins <= 256), "apsp_bfs_batched: nbins %d out of [2,256]", nbins);
    if (max_n < 1 || max_n > GNAN_APSP_BATCHED_MAX_NODES) {
        gnan_set_error("apsp_bfs_batched: graphs with %d nodes unsupported (1..%d = GNAN_APSP_BATCHED_MAX_NODES); use gnan_apsp_bfs",
                       max_n, GNAN_APSP_BATCHED_MAX_NODES);
        return GNAN_ERR_UNSUPPORTED;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const bool levels = cnt || rscale;
    const int nb = levels ? nbins : 256;
    int rc = classify_by_size(node_off, B, max_n, order_ws, st);
    if (rc != GNAN_OK) return rc;
    rc = launch_bv3<false>(rowptr, col, node_off, hop_off, B, std::min(max_n, 32 * BV3_MAX_W), hop, cnt, rscale, nb, levels,
                           overflow_flag, max_level, order_ws, Bv3Edges{}, st);
    if (rc == GNAN_ERR_UNSUPPORTED) gnan_set_error("apsp_bfs_batched: level table too wide for the shared-memory slice");
    if (rc != GNAN_OK || max_n <= 32 * BV3_MAX_W) return rc;
    return launch_batched_large(rowptr, col, node_off, hop_off, B, hop, cnt, rscale, nb, overflow_flag, max_level, order_ws, st);
}

// The batched BFS straight from the batch's edge list in its transfer form (no CSR): see include/gnan_b200.h
extern "C" int gnan_apsp_bfs_batched_local(const uint8_t *src, const uint8_t *dst, const int32_t *edge_off, const int32_t *node_off,
                                           const int64_t *hop_off, int32_t B, int32_t max_n, uint8_t *hop, int32_t *cnt, float *rscale,
                                           int32_t nbins, int32_t *status, int32_t *overflow_flag, int32_t *max_level, int32_t *order_ws,
                                           gnan_stream_t stream)
{
    GNAN_REQUIRE(B >= 0, "apsp_bfs_batched_local: negative batch");
    GNAN_REQUIRE(status != nullptr, "apsp_bfs_batched_local: NULL status");
    cudaStream_t st = (cudaStream_t)stream;
    GNAN_CUDA(cudaMemsetAsync(status, 0, sizeof(int32_t), st));
    if (B == 0) return GNAN_OK;
    GNAN_REQUIRE(edge_off && node_off && hop_off && hop && overflow_flag && order_ws, "apsp_bfs_batched_local: NULL pointer");
    GNAN_REQUIRE(!(cnt || rscale) || (nbins >= 2 && nbins <= 256), "apsp_bfs_batched_local: nbins %d out of [2,256]", nbins);
    if (max_n < 1 || max_n > 32 * BV3_MAX_W) {
        gnan_set_error("apsp_bfs_batched_local: graphs with %d nodes unsupported (1..%d); expand the edges and use gnan_apsp_bfs_batched_ex",
                       max_n, 32 * BV3_MAX_W);
        return GNAN_ERR_UNSUPPORTED;
    }
    const bool levels = cnt || rscale;
    const Bv3Edges le{src, dst, edge_off, status};
    int rc = classify_by_size(node_off, B, max_n, order_ws, st);
    if (rc != GNAN_OK) return rc;
    rc = launch_bv3<true>(nullptr, nullptr, node_off, hop_off, B, max_n, hop, cnt, rscale, levels ? nbins : 256, levels,
                          overflow_flag, max_level, order_ws, le, st);
    if (rc == GNAN_ERR_UNSUPPORTED) gnan_set_error("apsp_bfs_batched_local: level table too wide for the shared-memory slice");
    return rc;
}

// graphs of more than 128 nodes of a fused readout batch: class 4 of order_ws [5*B+5], one CTA each, sized by max_n
template <typename IT, int CC>
static int launch_readout_large(Bv3EdgesT<IT> le, const int32_t *node_off, int32_t B, int32_t max_n, int nbins, const Bv3Readout &ro,
                                int32_t *overflow_flag, int32_t *max_level, const int32_t *order_ws, cudaStream_t st)
{
    const int nt = brl_threads(max_n);
    const size_t smem = brl_need(max_n, nt, nbins, CC);
    auto kernel = bfs_readout_large_kernel<IT, CC>;
    static thread_local size_t cached_smem = 0;
    static thread_local int cached_nt = 0, per_sm = 0;
    if (cached_smem != smem || cached_nt != nt || per_sm == 0) {
        GNAN_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        GNAN_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, nt, smem));
        cached_smem = smem; cached_nt = nt;
    }
    if (per_sm < 1) return GNAN_ERR_UNSUPPORTED;
    const int blocks = (int)std::min<int64_t>(B, (int64_t)per_sm * gnan_sm_count());
    kernel<<<blocks, nt, smem, st>>>(le.src, le.dst, le.edge_off, node_off, B, max_n, nbins, ro, le.status, overflow_flag, max_level,
                                     order_ws);
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}

// The batched BFS fused with the output-normalised graph readout, straight from the batch's edge list: graphs of at most 128 nodes
// on the v3 kernel, larger ones (up to max_cap) on bfs_readout_large_kernel. See include/gnan_b200.h
template <typename IT>
static int bfs_graph_readout(const char *who, int max_cap, const IT *src, const IT *dst, const int32_t *edge_off, const int32_t *node_off,
                             int32_t B, int32_t max_n, int32_t nbins, const float *T, int32_t Cr, const float *S, int32_t C, float *out,
                             float *colw, float *Q, int32_t *status, int32_t *overflow_flag, int32_t *max_level, int32_t *order_ws,
                             cudaStream_t st)
{
    GNAN_REQUIRE(B >= 0, "%s: negative batch", who);
    GNAN_REQUIRE(status != nullptr, "%s: NULL status", who);
    if (!gnan_aggregate_blockdiag_graph_supported(nbins, Cr, C)) {
        gnan_set_error("%s: needs 2 <= nbins <= 64, C <= 4, Cr in {1,C} (nbins=%d Cr=%d C=%d)", who, nbins, Cr, C);
        return GNAN_ERR_UNSUPPORTED;
    }
    if (B > 0 && (max_n < 1 || max_n > max_cap)) {
        gnan_set_error("%s: graphs with %d nodes unsupported (1..%d)", who, max_n, max_cap);
        return GNAN_ERR_UNSUPPORTED;
    }
    GNAN_CUDA(cudaMemsetAsync(status, 0, sizeof(int32_t), st));
    if (B == 0) return GNAN_OK;
    // src / dst are read only inside the graphs' edge segments: NULL is fine for a batch without edges (an empty edge list)
    GNAN_REQUIRE(edge_off && node_off && T && S && out && colw && Q && overflow_flag && order_ws, "%s: NULL pointer", who);
    const Bv3EdgesT<IT> le{src, dst, edge_off, status};
    const Bv3Readout ro{T, S, Cr, C, out, colw, Q};
    const int small_n = std::min(max_n, 32 * BV3_MAX_W);
    auto launch = [&](auto cc) {
        constexpr int CC = decltype(cc)::value;
        int rc = launch_bv3<true, CC, IT>(nullptr, nullptr, node_off, nullptr, B, small_n, nullptr, nullptr, nullptr, nbins, false,
                                          overflow_flag, max_level, order_ws, le, st, ro);
        if (rc == GNAN_OK && max_n > 32 * BV3_MAX_W)
            rc = launch_readout_large<IT, CC>(le, node_off, B, max_n, nbins, ro, overflow_flag, max_level, order_ws, st);
        return rc;
    };
    int rc = classify_by_size(node_off, B, max_n, order_ws, st);
    if (rc != GNAN_OK) return rc;
    rc = C == 1 ? launch(std::integral_constant<int, 1>{}) : C == 2 ? launch(std::integral_constant<int, 2>{})
                                                                   : launch(std::integral_constant<int, 4>{});
    if (rc == GNAN_ERR_UNSUPPORTED) gnan_set_error("%s: per-graph state too large for shared memory", who);
    return rc;
}

extern "C" int gnan_bfs_graph_readout_fwd(const uint8_t *src, const uint8_t *dst, const int32_t *edge_off, const int32_t *node_off,
                                          int32_t B, int32_t max_n, int32_t nbins, const float *T, int32_t Cr, const float *S, int32_t C,
                                          float *out, float *colw, float *Q, int32_t *status, int32_t *overflow_flag, int32_t *max_level,
                                          int32_t *order_ws, gnan_stream_t stream)
{
    return bfs_graph_readout<uint8_t>("bfs_graph_readout_fwd", 256, src, dst, edge_off, node_off, B, max_n, nbins, T, Cr, S, C, out,
                                      colw, Q, status, overflow_flag, max_level, order_ws, (cudaStream_t)stream);
}

extern "C" int gnan_bfs_graph_readout_fwd_i16(const int16_t *src, const int16_t *dst, const int32_t *edge_off, const int32_t *node_off,
                                              int32_t B, int32_t max_n, int32_t nbins, const float *T, int32_t Cr, const float *S,
                                              int32_t C, float *out, float *colw, float *Q, int32_t *status, int32_t *overflow_flag,
                                              int32_t *max_level, int32_t *order_ws, gnan_stream_t stream)
{
    return bfs_graph_readout<int16_t>("bfs_graph_readout_fwd_i16", GNAN_APSP_BATCHED_MAX_NODES, src, dst, edge_off, node_off, B, max_n,
                                      nbins, T, Cr, S, C, out, colw, Q, status, overflow_flag, max_level, order_ws, (cudaStream_t)stream);
}

extern "C" int gnan_hops_to_reference(const uint8_t *hop, int64_t R, int64_t N, int64_t ld_hop, const int32_t *cnt,
                                      int32_t nbins, float *node_distances, float *normalization_matrix, gnan_stream_t stream)
{
    GNAN_REQUIRE(R >= 0 && N >= 0 && ld_hop >= N, "hops_to_reference: bad shape");
    if (R * N == 0) return GNAN_OK;
    GNAN_REQUIRE(hop && (node_distances || normalization_matrix), "hops_to_reference: NULL pointer");
    GNAN_REQUIRE(!normalization_matrix || (cnt && nbins >= 2), "hops_to_reference: cnt required for the normalisation matrix");
    hops_to_reference_kernel<<<(unsigned)ceil_div64(R * N, 256), 256, 0, (cudaStream_t)stream>>>(hop, R, N, ld_hop, cnt, nbins,
                                                                                                  node_distances, normalization_matrix);
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}

extern "C" int gnan_hops_from_reference(const float *node_distances, const float *normalization_matrix, int64_t R, int64_t N,
                                        uint8_t *hop, int64_t ld_hop, int32_t *cnt, int32_t nbins, int32_t *overflow_flag,
                                        gnan_stream_t stream)
{
    GNAN_REQUIRE(R >= 0 && N >= 0 && ld_hop >= N, "hops_from_reference: bad shape");
    if (R * N == 0) return GNAN_OK;
    GNAN_REQUIRE(node_distances && hop && overflow_flag, "hops_from_reference: NULL pointer");
    GNAN_REQUIRE(nbins >= 2 && nbins <= 256, "hops_from_reference: nbins %d out of [2,256]", nbins);
    hops_from_reference_kernel<<<(unsigned)ceil_div64(R * ld_hop, 256), 256, 0, (cudaStream_t)stream>>>(
        node_distances, normalization_matrix, R, N, hop, ld_hop, cnt, nbins, overflow_flag);
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}
