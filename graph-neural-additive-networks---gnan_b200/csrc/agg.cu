// Distance-table aggregation over uint8 hop matrices (dense row blocks and block-diagonal batches).
//
// Reference lines replaced: GNAN.py:65-79 (rho on N*N pairs, permute, bmm, sums), GNAN.py:159-170 (row loop),
// models.py:366-384, batched_pyg_main.py:154-181; backward = autograd through the same.
//
//   out[i,c] = sum_j W[i,j,c] S[j,c],  W[i,j,c] = T[ti, b(hop[i,j]), c'] * rscale[i, b(hop[i,j])]
//
// The N*N rho evaluation of the reference is a lookup into a (per-row or global) table with nbins = D+2 rows.
// HBM traffic is the hop bytes: 1 B per ordered pair per pass; one pass forward, one pass backward.
//
// Forward (agg_rows_bins_kernel): row-stationary. A warp owns a row and keeps lane-private bin sums
// Bsum[i,d,c] = sum_{j: b(hop[i,j])=d} S[j,c] in shared memory (conflict-free layout), so the pass is adds only; the table is
// applied once per row at the end. Bsum is also what the backward needs for dT, so it is saved (N*nbins*C floats).
// Backward (agg_rows_ds_kernel): column-stationary. A thread owns 16 columns, keeps dS[j,c] in registers and walks down
// its rows, looking up the pre-multiplied table TG[i][d][c] = W-table * g[i,c] staged in shared memory.
#include <algorithm>

#include "common.cuh"

namespace {

constexpr int BINS_WARPS = 8;       // warps per CTA in the bins kernel (may be lowered to fit smem)
constexpr int CHUNK_FLOATS = 4096;  // floats of S staged per sweep step: 4096 / CC columns
constexpr int DS_THREADS = 256;
constexpr int DS_RB = 8;            // rows per staged table group in the dS kernel

template <int CC> struct VecT;
template <> struct VecT<1> { using type = float; };
template <> struct VecT<2> { using type = float2; };
template <> struct VecT<4> { using type = float4; };

__device__ __forceinline__ void vadd(float &a, const float &b) { a += b; }
__device__ __forceinline__ void vadd(float2 &a, const float2 &b) { a.x += b.x; a.y += b.y; }
__device__ __forceinline__ void vadd(float4 &a, const float4 &b) { a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }
__device__ __forceinline__ void vzero(float &a) { a = 0.f; }
__device__ __forceinline__ void vzero(float2 &a) { a = make_float2(0.f, 0.f); }
__device__ __forceinline__ void vzero(float4 &a) { a = make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ float vget(const float &a, int) { return a; }
__device__ __forceinline__ float vget(const float2 &a, int i) { return i == 0 ? a.x : a.y; }
__device__ __forceinline__ float vget(const float4 &a, int i) { return i == 0 ? a.x : i == 1 ? a.y : i == 2 ? a.z : a.w; }
__device__ __forceinline__ void vset(float &a, int, float v) { a = v; }
__device__ __forceinline__ void vset(float2 &a, int i, float v) { if (i == 0) a.x = v; else a.y = v; }
__device__ __forceinline__ void vset(float4 &a, int i, float v) { if (i == 0) a.x = v; else if (i == 1) a.y = v; else if (i == 2) a.z = v; else a.w = v; }

struct AggArgs {
    const uint8_t *hop;
    int64_t R, N, ld;
    const float *T;       // [nbins,Cr] or [R,nbins,Cr]
    int per_row, nbins, Cr;
    const float *rscale;  // [R,nbins] or NULL
    const float *S;       // [N,C]
    int C;
};

__device__ __forceinline__ float table_value(const AggArgs &a, int64_t i, int d, int c)
{
    const int cr = a.Cr == 1 ? 0 : c;
    const float t = a.per_row ? a.T[(i * a.nbins + d) * a.Cr + cr] : a.T[d * a.Cr + cr];
    return a.rscale ? t * a.rscale[i * a.nbins + d] : t;
}

// ---- forward: bins --------------------------------------------------------------------------------------------
// grid (row groups, channel chunks). Each warp: one row at a time; all warps sweep the same S chunk.
// WAYS independent lane-private bin arrays break the load-add-store dependency chain of consecutive pairs
template <int CC, int WAYS>
__global__ void __launch_bounds__(BINS_WARPS * 32)
agg_rows_bins_kernel(AggArgs a, int nwarps, float *__restrict__ out, float *__restrict__ Bsum)
{
    using V = typename VecT<CC>::type;
    constexpr int CHUNK = CHUNK_FLOATS / CC;
    constexpr int SROW = CHUNK / 16 + 2;                       // +2: the transposing stash (lane -> (t&15, t>>4)) is conflict-free
    extern __shared__ __align__(16) float smem[];
    V *sS = reinterpret_cast<V *>(smem);                       // [16][SROW]  permuted: column t of the chunk at (t%16, t/16)
    V *sBins = sS + 16 * SROW;                                 // [nwarps][ways][nbins][32]
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int c0 = blockIdx.y * CC;
    const bool active_warp = w < nwarps;
    const int64_t i = (int64_t)blockIdx.x * nwarps + w;
    const bool has_row = active_warp && i < a.R;
    const int way_stride = a.nbins * 32;                         // [way][bin][lane]
    V *bins = sBins + (size_t)w * WAYS * way_stride;
    if (active_warp)
        for (int d = 0; d < WAYS * a.nbins; ++d) vzero(bins[d * 32 + lane]);
    const uint8_t *hrow = a.hop + (has_row ? i : 0) * a.ld;

    // S chunks are double-buffered through registers: the next chunk's global loads are in flight while the current chunk is
    // consumed from shared memory (their L2 latency used to be exposed at every chunk barrier)
    constexpr int PER_T = CHUNK / (BINS_WARPS * 32);
    V nxt[PER_T];
    auto fetch = [&](int64_t jb) {
#pragma unroll
        for (int k = 0; k < PER_T; ++k) {
            const int64_t j = jb + threadIdx.x + k * (BINS_WARPS * 32);
            V v;
            vzero(v);
            if (j < a.N) {
#pragma unroll
                for (int cc = 0; cc < CC; ++cc)
                    if (c0 + cc < a.C) vset(v, cc, __ldg(a.S + j * a.C + c0 + cc));
            }
            nxt[k] = v;
        }
    };
    auto stash = [&]() {
#pragma unroll
        for (int k = 0; k < PER_T; ++k) {
            const int t = threadIdx.x + k * (BINS_WARPS * 32);
            sS[(t & 15) * SROW + (t >> 4)] = nxt[k];
        }
    };
    fetch(0);
    stash();
    __syncthreads();
    for (int64_t jb = 0; jb < a.N; jb += CHUNK) {
        const bool more = jb + CHUNK < a.N;
        if (more) fetch(jb + CHUNK);
        if (has_row) {
            const int len = (int)min((int64_t)CHUNK, a.N - jb);
            const int nb1 = a.nbins - 1;
            V *mybins = bins + lane;                             // bin b of this lane lives at mybins[b * 32]
            uint4 hv_n = make_uint4(0u, 0u, 0u, 0u);
            if (lane * 16 < len) hv_n = __ldcs(reinterpret_cast<const uint4 *>(hrow + jb + lane * 16));
            for (int j0 = lane * 16; j0 < len; j0 += 512) {
                const uint4 hv = hv_n;                           // hop bytes are fetched one step ahead (more bytes in flight)
                if (j0 + 512 < len) hv_n = __ldcs(reinterpret_cast<const uint4 *>(hrow + jb + j0 + 512));
                const uint32_t hw[4] = {hv.x, hv.y, hv.z, hv.w};
                const V *sp = sS + (j0 >> 4);                    // S of column j0 + q sits at sp[q * SROW]
                if (j0 + 16 <= len) {                            // fast path: 16 pairs, no bounds checks, WAYS pairs in flight
#pragma unroll
                    for (int q = 0; q < 16; q += WAYS) {
                        int b[WAYS];
                        V cur[WAYS];
#pragma unroll
                        for (int u = 0; u < WAYS; ++u) {
                            const int h = (int)__byte_perm(hw[(q + u) >> 2], 0u, 0x4440u + ((q + u) & 3));
                            b[u] = min(h, nb1) * 32 + u * way_stride;
                            cur[u] = mybins[b[u]];
                        }
#pragma unroll
                        for (int u = 0; u < WAYS; ++u) vadd(cur[u], sp[(q + u) * SROW]);
#pragma unroll
                        for (int u = 0; u < WAYS; ++u) mybins[b[u]] = cur[u];
                    }
                } else {
#pragma unroll
                    for (int q = 0; q < 16; ++q) {
                        if (j0 + q < len) {
                            const int h = (int)__byte_perm(hw[q >> 2], 0u, 0x4440u + (q & 3));
                            const int b = min(h, nb1);
                            V cur = mybins[b * 32];
                            vadd(cur, sp[q * SROW]);
                            mybins[b * 32] = cur;
                        }
                    }
                }
            }
        }
        __syncthreads();                 // everyone is done with the current chunk
        if (more) stash();
        __syncthreads();
    }
    if (!has_row) return;
    __syncwarp();
    // reduce lane-private bins: lane handles bin d = lane, lane+32, ...
    float o[CC];
#pragma unroll
    for (int cc = 0; cc < CC; ++cc) o[cc] = 0.f;
    for (int d = lane; d < a.nbins; d += 32) {
        V tot;
        vzero(tot);
        for (int u = 0; u < WAYS; ++u)
            for (int k = 0; k < 32; ++k) vadd(tot, bins[u * way_stride + d * 32 + ((k + lane) & 31)]);
#pragma unroll
        for (int cc = 0; cc < CC; ++cc)
            if (c0 + cc < a.C) {
                const float bs = vget(tot, cc);
                if (Bsum) Bsum[(i * a.nbins + d) * a.C + c0 + cc] = bs;
                o[cc] = fmaf(table_value(a, i, d, c0 + cc), bs, o[cc]);
            }
    }
#pragma unroll
    for (int cc = 0; cc < CC; ++cc) {
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) o[cc] += __shfl_xor_sync(0xffffffffu, o[cc], s);
        if (lane == 0 && c0 + cc < a.C) out[i * a.C + c0 + cc] = o[cc];
    }
}

// ---- backward: dS ---------------------------------------------------------------------------------------------
// grid (column chunks of 256*16, row super-blocks, channel chunks); dSpart[sb][N][C]
template <int CC>
__global__ void __launch_bounds__(DS_THREADS)
agg_rows_ds_kernel(AggArgs a, const float *__restrict__ g, int64_t rows_per_sb, float *__restrict__ dSpart)
{
    using V = typename VecT<CC>::type;
    extern __shared__ __align__(16) float smem[];
    V *sTG = reinterpret_cast<V *>(smem);  // [DS_RB][nbins]
    const int c0 = blockIdx.z * CC;
    const int64_t j0 = ((int64_t)blockIdx.x * DS_THREADS + threadIdx.x) * 16;
    const int64_t r_begin = (int64_t)blockIdx.y * rows_per_sb;
    const int64_t r_end = min(a.R, r_begin + rows_per_sb);
    const bool col_ok = j0 < a.ld;   // 16 bytes readable (ld is a multiple of 16)
    V acc[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) vzero(acc[q]);

    for (int64_t rb = r_begin; rb < r_end; rb += DS_RB) {
        const int nr = (int)min((int64_t)DS_RB, r_end - rb);
        __syncthreads();
        for (int t = threadIdx.x; t < nr * a.nbins; t += DS_THREADS) {
            const int r = t / a.nbins, d = t % a.nbins;
            const int64_t i = rb + r;
            V v;
            vzero(v);
#pragma unroll
            for (int cc = 0; cc < CC; ++cc)
                if (c0 + cc < a.C) vset(v, cc, table_value(a, i, d, c0 + cc) * __ldg(g + i * a.C + c0 + cc));
            sTG[r * a.nbins + d] = v;
        }
        __syncthreads();
        if (col_ok) {
            uint4 hv[DS_RB];
#pragma unroll
            for (int r = 0; r < DS_RB; ++r)
                if (r < nr) hv[r] = __ldcs(reinterpret_cast<const uint4 *>(a.hop + (rb + r) * a.ld + j0));
#pragma unroll
            for (int r = 0; r < DS_RB; ++r) {
                if (r < nr) {
                    const uint32_t hw[4] = {hv[r].x, hv[r].y, hv[r].z, hv[r].w};
                    const V *tg = sTG + r * a.nbins;
#pragma unroll
                    for (int q = 0; q < 16; ++q) {
                        const int h = (hw[q >> 2] >> ((q & 3) * 8)) & 0xff;
                        vadd(acc[q], tg[min(h, a.nbins - 1)]);
                    }
                }
            }
        }
    }
    float *dst = dSpart + (size_t)blockIdx.y * a.N * a.C;
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        const int64_t j = j0 + q;
        if (j < a.N) {
#pragma unroll
            for (int cc = 0; cc < CC; ++cc)
                if (c0 + cc < a.C) dst[j * a.C + c0 + cc] = vget(acc[q], cc);
        }
    }
}

// dT from the saved bin sums.  per-row: dT[i,d,cr] = rs[i,d] * sum_c g[i,c] Bsum[i,d,c]   (elementwise over (i,d))
__global__ void agg_dt_per_row_kernel(AggArgs a, const float *__restrict__ g, const float *__restrict__ Bsum,
                                      float *__restrict__ dT)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= a.R * a.nbins) return;
    const int64_t i = t / a.nbins;
    const float rs = a.rscale ? a.rscale[t] : 1.f;
    if (a.Cr == 1) {
        float s = 0.f;
        for (int c = 0; c < a.C; ++c) s = fmaf(g[i * a.C + c], Bsum[t * a.C + c], s);
        dT[t] = s * rs;
    } else {
        for (int c = 0; c < a.C; ++c) dT[t * a.C + c] = g[i * a.C + c] * Bsum[t * a.C + c] * rs;
    }
}

// global table: dT[d,cr] = sum_i rs[i,d] sum_c g[i,c] Bsum[i,d,c]; thread <-> (d,c), CTA <-> row slab; atomics at the end
__global__ void agg_dt_global_kernel(AggArgs a, const float *__restrict__ g, const float *__restrict__ Bsum,
                                     int64_t rows_per_cta, float *__restrict__ dT)
{
    const int64_t r0 = (int64_t)blockIdx.x * rows_per_cta, r1 = min(a.R, r0 + rows_per_cta);
    const int E = a.nbins * a.C;
    for (int e = threadIdx.x; e < E; e += blockDim.x) {
        const int d = e / a.C, c = e % a.C;
        float s = 0.f;
        for (int64_t i = r0; i < r1; ++i) {
            const float rs = a.rscale ? a.rscale[i * a.nbins + d] : 1.f;
            s = fmaf(g[i * a.C + c] * rs, Bsum[i * E + e], s);
        }
        atomicAdd(dT + d * a.Cr + (a.Cr == 1 ? 0 : c), s);
    }
}

// ---- block-diagonal batches ------------------------------------------------------------------------------------
struct BdArgs {
    const uint8_t *hop;
    const int64_t *hop_off;
    const int32_t *node_off;
    int B;
    const float *T;
    int per_row, nbins, Cr;
    const float *rscale;
    const float *S;
    int C;
    int reduce_graph;
};

__device__ __forceinline__ float bd_table(const BdArgs &a, int64_t node, int d, int c)
{
    const int cr = a.Cr == 1 ? 0 : c;
    const float t = a.per_row ? a.T[(node * a.nbins + d) * a.Cr + cr] : a.T[d * a.Cr + cr];
    return a.rscale ? t * a.rscale[node * a.nbins + d] : t;
}

// one warp per graph (grid-stride over graphs); lanes stride over columns j.
__global__ void __launch_bounds__(256)
agg_blockdiag_fwd_kernel(BdArgs a, float *__restrict__ out)
{
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t b = warp; b < a.B; b += nwarps) {
        const int n0 = a.node_off[b], n = a.node_off[b + 1] - n0;
        const uint8_t *hb = a.hop + a.hop_off[b];
        for (int c = 0; c < a.C; ++c) {
            float gsum = 0.f;
            for (int i = 0; i < n; ++i) {
                float acc = 0.f;
                for (int j = lane; j < n; j += 32) {
                    const int d = min((int)hb[(size_t)i * n + j], a.nbins - 1);
                    acc = fmaf(bd_table(a, n0 + i, d, c), a.S[(int64_t)(n0 + j) * a.C + c], acc);
                }
#pragma unroll
                for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
                if (a.reduce_graph) gsum += acc;
                else if (lane == 0) out[(int64_t)(n0 + i) * a.C + c] = acc;
            }
            if (a.reduce_graph && lane == 0) out[b * a.C + c] = gsum;
        }
    }
}

// v2 forward: one warp per graph, a lane owns ROWS i = lane, lane+32, .. and walks its own hop row (consecutive bytes of one
// 32-byte sector: served by L1 after the first touch; the n x n block is at most 64 KB). All loads of a row are independent,
// so many are in flight per lane, and nothing is reduced across lanes until the per-graph sum at the very end (the v1 kernel
// paid a 5-step shuffle chain behind a dependent global load for every row). S[j,:] is a broadcast load.
template <int CC>
__global__ void __launch_bounds__(256)
agg_blockdiag_fwd_rows_kernel(BdArgs a, float *__restrict__ out)
{
    extern __shared__ float sT[];                      // global table copy [nbins*Cr]
    const int lane = threadIdx.x & 31;
    if (!a.per_row) {
        for (int t = threadIdx.x; t < a.nbins * a.Cr; t += blockDim.x) sT[t] = a.T[t];
        __syncthreads();
    }
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int nb1 = a.nbins - 1;
    for (int64_t b = warp; b < a.B; b += nwarps) {
        const int n0 = a.node_off[b], n = a.node_off[b + 1] - n0;
        const uint8_t *hb = a.hop + a.hop_off[b];
        for (int c0 = 0; c0 < a.C; c0 += CC) {
            float gsum[CC];
#pragma unroll
            for (int cc = 0; cc < CC; ++cc) gsum[cc] = 0.f;
            for (int i = lane; i < n; i += 32) {
                const uint8_t *row = hb + (size_t)i * n;
                const float *Ti = a.per_row ? a.T + (int64_t)(n0 + i) * a.nbins * a.Cr : sT;
                const float *rsi = a.rscale ? a.rscale + (int64_t)(n0 + i) * a.nbins : nullptr;
                float acc[CC];
#pragma unroll
                for (int cc = 0; cc < CC; ++cc) acc[cc] = 0.f;
#pragma unroll 4
                for (int j = 0; j < n; ++j) {
                    const int d = min((int)row[j], nb1);
                    const float r = rsi ? rsi[d] : 1.f;
                    const float *Sj = a.S + (int64_t)(n0 + j) * a.C + c0;
#pragma unroll
                    for (int cc = 0; cc < CC; ++cc)
                        if (c0 + cc < a.C) acc[cc] = fmaf(Ti[d * a.Cr + (a.Cr == 1 ? 0 : c0 + cc)] * r, Sj[cc], acc[cc]);
                }
#pragma unroll
                for (int cc = 0; cc < CC; ++cc) {
                    if (a.reduce_graph) gsum[cc] += acc[cc];
                    else if (c0 + cc < a.C) out[(int64_t)(n0 + i) * a.C + c0 + cc] = acc[cc];
                }
            }
            if (a.reduce_graph) {
#pragma unroll
                for (int cc = 0; cc < CC; ++cc) {
                    float v = gsum[cc];
#pragma unroll
                    for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
                    if (lane == 0 && c0 + cc < a.C) out[b * a.C + c0 + cc] = v;
                }
            }
        }
    }
}

// backward: dS (lane owns column j), dT via shared-memory bins (per CTA for a global table, per row otherwise)
__global__ void __launch_bounds__(256)
agg_blockdiag_bwd_kernel(BdArgs a, const float *__restrict__ g, float *__restrict__ dS, float *__restrict__ dT)
{
    extern __shared__ float sb[];  // global table: [nbins*Cr] CTA-wide ; per-row: [8 warps][nbins*Cr]
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int nT = a.nbins * a.Cr;
    float *bins = a.per_row ? sb + w * nT : sb;
    if (!a.per_row) {
        for (int t = threadIdx.x; t < nT; t += blockDim.x) sb[t] = 0.f;
        __syncthreads();
    }
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t b = warp; b < a.B; b += nwarps) {
        const int n0 = a.node_off[b], n = a.node_off[b + 1] - n0;
        const uint8_t *hb = a.hop + a.hop_off[b];
        // dS[j,c] = sum_i W[i,j,c] g_i[c]
        for (int j = lane; j < n; j += 32) {
            for (int c = 0; c < a.C; ++c) {
                float acc = 0.f;
                for (int i = 0; i < n; ++i) {
                    const int d = min((int)hb[(size_t)i * n + j], a.nbins - 1);
                    const float gi = a.reduce_graph ? g[b * a.C + c] : g[(int64_t)(n0 + i) * a.C + c];
                    acc = fmaf(bd_table(a, n0 + i, d, c), gi, acc);
                }
                dS[(int64_t)(n0 + j) * a.C + c] = acc;
            }
        }
        // dT
        for (int i = 0; i < n; ++i) {
            if (a.per_row) {
                for (int t = lane; t < nT; t += 32) bins[t] = 0.f;
                __syncwarp();
            }
            for (int j = lane; j < n; j += 32) {
                const int d = min((int)hb[(size_t)i * n + j], a.nbins - 1);
                const float rs = a.rscale ? a.rscale[(int64_t)(n0 + i) * a.nbins + d] : 1.f;
                for (int c = 0; c < a.C; ++c) {
                    const float gi = a.reduce_graph ? g[b * a.C + c] : g[(int64_t)(n0 + i) * a.C + c];
                    atomicAdd(bins + d * a.Cr + (a.Cr == 1 ? 0 : c), rs * gi * a.S[(int64_t)(n0 + j) * a.C + c]);
                }
            }
            if (a.per_row) {
                __syncwarp();
                for (int t = lane; t < nT; t += 32) dT[(int64_t)(n0 + i) * nT + t] = bins[t];
                __syncwarp();
            }
        }
    }
    if (!a.per_row) {
        __syncthreads();
        for (int t = threadIdx.x; t < nT; t += blockDim.x)
            if (sb[t] != 0.f) atomicAdd(dT + t, sb[t]);
    }
}

// backward for a GLOBAL table (models.py TensorGNAN, batched variant): one pass over the pairs gives both gradients, no atomics
// in the pair loop. A lane owns columns j = lane, lane+32, ..: dS[j] accumulates in a register; dT accumulates in a lane-private
// shared-memory column accT[t][lane] that persists over all graphs of the warp and is reduced over lanes once at the end.
__global__ void __launch_bounds__(256)
agg_blockdiag_bwd_global_kernel(BdArgs a, const float *__restrict__ g, float *__restrict__ dS, float *__restrict__ dT)
{
    extern __shared__ float sb[];                      // [nT] table copy, then [8 warps][nT][32] accumulators
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int nT = a.nbins * a.Cr;
    float *sT = sb;
    float *acc = sb + nT + (size_t)w * nT * 32;
    for (int t = threadIdx.x; t < nT; t += blockDim.x) sT[t] = a.T[t];
    for (int t = lane; t < nT * 32; t += 32) acc[t] = 0.f;
    __syncthreads();
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t b = warp; b < a.B; b += nwarps) {
        const int n0 = a.node_off[b], n = a.node_off[b + 1] - n0;
        const uint8_t *hb = a.hop + a.hop_off[b];
        for (int c = 0; c < a.C; ++c) {
            const int cr = a.Cr == 1 ? 0 : c;
            const float gb = a.reduce_graph ? g[b * a.C + c] : 0.f;
            for (int j = lane; j < n; j += 32) {
                const float sj = a.S[(int64_t)(n0 + j) * a.C + c];
                float ds = 0.f;
                for (int i0 = 0; i0 < n; i0 += 8) {
                    // 8 rows per step: their hop bytes and scale factors are all in flight before the first shared-memory
                    // update (one dependent global load per row used to be exposed in full)
                    int d[8];
                    float r[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) d[u] = i0 + u < n ? min((int)hb[(size_t)(i0 + u) * n + j], a.nbins - 1) : -1;
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        r[u] = 0.f;
                        if (d[u] >= 0) {
                            r[u] = a.reduce_graph ? gb : g[(int64_t)(n0 + i0 + u) * a.C + c];
                            if (a.rscale) r[u] *= a.rscale[(int64_t)(n0 + i0 + u) * a.nbins + d[u]];
                        }
                    }
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        if (d[u] >= 0) {
                            const int t = d[u] * a.Cr + cr;
                            ds = fmaf(sT[t], r[u], ds);
                            acc[t * 32 + lane] = fmaf(r[u], sj, acc[t * 32 + lane]);
                        }
                    }
                }
                dS[(int64_t)(n0 + j) * a.C + c] = ds;
            }
        }
    }
    __syncwarp();
    for (int t = 0; t < nT; ++t) {
        float v = acc[t * 32 + lane];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0 && v != 0.f) atomicAdd(dT + t, v);
    }
}

// ---- small helpers ---------------------------------------------------------------------------------------------
__global__ void rho_table_inputs_kernel(const int32_t *__restrict__ cnt, int64_t rows, int nbins, int raw, float *__restrict__ u)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t total = (rows > 0 ? rows : 1) * nbins;
    if (t >= total) return;
    const int d = (int)(t % nbins);
    float v;
    if (raw) v = (float)d;
    else v = d == nbins - 1 ? 0.f : 1.0f / ((float)d + 1.0f);   // fp32 division, as pre_process_datasets.py:113-114
    if (cnt && !raw) {
        const int c = cnt[t];
        v = c > 0 ? v / (float)c : 0.f;                          // GNAN.py:66 (empty bins are never gathered)
    }
    u[t] = v;
}

__global__ void level_rscale_kernel(const int32_t *__restrict__ cnt, int64_t total, float *__restrict__ rs)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const int c = cnt[t];
    rs[t] = c > 0 ? 1.0f / (float)c : 0.f;
}

int check_agg(const char *who, const uint8_t *hop, int64_t R, int64_t N, int64_t ld, const float *T, int nbins, int Cr,
              const float *S, int C)
{
    GNAN_REQUIRE(R >= 0 && N >= 0, "%s: negative shape", who);
    GNAN_REQUIRE(hop && T && S, "%s: NULL hop/T/S", who);
    GNAN_REQUIRE(ld >= N && ld % 16 == 0 && ((uintptr_t)hop % 16) == 0, "%s: hop rows must be 16-byte aligned with ld %% 16 == 0 (ld=%lld)", who, (long long)ld);
    GNAN_REQUIRE(nbins >= 2 && nbins <= 256, "%s: nbins %d out of [2,256]", who, nbins);
    GNAN_REQUIRE(C >= 1 && (Cr == 1 || Cr == C), "%s: Cr must be 1 or C (Cr=%d C=%d)", who, Cr, C);
    return GNAN_OK;
}

struct DsPlan { int nsb; int64_t rows_per_sb; int ncol; };
DsPlan plan_ds(int64_t R, int64_t N)
{
    DsPlan p;
    p.ncol = (int)ceil_div64(N, (int64_t)DS_THREADS * 16);
    int nsb = (int)ceil_div64(2 * gnan_sm_count() * 2, p.ncol);
    int64_t maxsb = ceil_div64(R, DS_RB);
    if (nsb > maxsb) nsb = (int)maxsb;
    if (nsb < 1) nsb = 1;
    p.rows_per_sb = ceil_div64(ceil_div64(R, nsb), DS_RB) * DS_RB;
    p.nsb = (int)ceil_div64(R, p.rows_per_sb);
    return p;
}

}  // namespace

extern "C" int gnan_rho_table_inputs(const int32_t *cnt, int64_t rows, int32_t nbins, int raw, float *u, gnan_stream_t stream)
{
    GNAN_REQUIRE(u && nbins >= 2 && rows >= 0, "rho_table_inputs: bad arguments");
    const int64_t total = (rows > 0 ? rows : 1) * nbins;
    rho_table_inputs_kernel<<<(unsigned)ceil_div64(total, 256), 256, 0, (cudaStream_t)stream>>>(rows > 0 ? cnt : nullptr, rows, nbins, raw, u);
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}

extern "C" int gnan_level_rscale(const int32_t *cnt, int64_t rows, int32_t nbins, float *rscale, gnan_stream_t stream)
{
    GNAN_REQUIRE(cnt && rscale && nbins >= 2 && rows >= 0, "level_rscale: bad arguments");
    if (rows == 0) return GNAN_OK;
    level_rscale_kernel<<<(unsigned)ceil_div64(rows * nbins, 256), 256, 0, (cudaStream_t)stream>>>(cnt, rows * nbins, rscale);
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}

// CUDA-core path of gnan_aggregate_rows_fwd_ws (agg_tc.cu), with optional Bsum save
int gnan_agg_rows_fwd_cuda_cores(const uint8_t *hop, int64_t R, int64_t N, int64_t ld_hop, const float *T, int table_per_row,
                                 int32_t nbins, int32_t Cr, const float *rscale, const float *S, int32_t C, float *out, float *Bsum,
                                 gnan_stream_t stream)
{
    int rc = check_agg("aggregate_rows_fwd", hop, R, N, ld_hop, T, nbins, Cr, S, C);
    if (rc) return rc;
    GNAN_REQUIRE(out != nullptr, "aggregate_rows_fwd: NULL out");
    if (R == 0) return GNAN_OK;
    cudaStream_t st = (cudaStream_t)stream;
    AggArgs a{hop, R, N, ld_hop, T, table_per_row, nbins, Cr, rscale, S, C};
    const int CC = C >= 4 ? 4 : (C >= 2 ? 2 : 1);
    const int WAYS = 2;
    int nwarps = BINS_WARPS;
    auto smem_of = [&](int nw) { return sizeof(float) * ((size_t)CHUNK_FLOATS + 32 * CC + (size_t)CC * nw * WAYS * nbins * 32); };
    while (nwarps > 1 && smem_of(nwarps) > 100 * 1024) nwarps >>= 1;   // keep >= 2 CTAs per SM
    if (smem_of(nwarps) > 227 * 1024) {
        gnan_set_error("aggregate_rows_fwd: nbins %d too large for shared memory", nbins);
        return GNAN_ERR_UNSUPPORTED;
    }
    const size_t smem = smem_of(nwarps);
    dim3 grid((unsigned)ceil_div64(R, nwarps), (unsigned)((C + CC - 1) / CC));
    if (CC == 4) {
        GNAN_CUDA(cudaFuncSetAttribute(agg_rows_bins_kernel<4, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        agg_rows_bins_kernel<4, 2><<<grid, BINS_WARPS * 32, smem, st>>>(a, nwarps, out, Bsum);
    } else if (CC == 2) {
        GNAN_CUDA(cudaFuncSetAttribute(agg_rows_bins_kernel<2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        agg_rows_bins_kernel<2, 2><<<grid, BINS_WARPS * 32, smem, st>>>(a, nwarps, out, Bsum);
    } else {
        GNAN_CUDA(cudaFuncSetAttribute(agg_rows_bins_kernel<1, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        agg_rows_bins_kernel<1, 2><<<grid, BINS_WARPS * 32, smem, st>>>(a, nwarps, out, Bsum);
    }
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}

size_t gnan_agg_rows_bwd_cuda_cores_bytes(int64_t R, int64_t N, int32_t nbins, int32_t C)
{
    if (R <= 0 || N <= 0) return 0;
    const DsPlan p = plan_ds(R, N);
    // [nsb][N][C] dS partials + [R][nbins][C] bin sums (recomputed when the caller did not save them)
    return sizeof(float) * ((size_t)p.nsb * N * C + (size_t)R * nbins * C);
}

// CUDA-core path of gnan_aggregate_rows_bwd_ws (agg_tc.cu), given saved Bsum (may be NULL -> recomputed into the workspace with
// one extra pass)
int gnan_agg_rows_bwd_cuda_cores(const uint8_t *hop, int64_t R, int64_t N, int64_t ld_hop, const float *T, int table_per_row,
                                 int32_t nbins, int32_t Cr, const float *rscale, const float *S, int32_t C, const float *g,
                                 const float *Bsum, float *dS, float *dT, void *workspace, size_t workspace_bytes,
                                 gnan_stream_t stream)
{
    int rc = check_agg("aggregate_rows_bwd", hop, R, N, ld_hop, T, nbins, Cr, S, C);
    if (rc) return rc;
    GNAN_REQUIRE(g || R == 0, "aggregate_rows_bwd: NULL g");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t nT = (size_t)(table_per_row ? R : 1) * nbins * Cr;
    if (R == 0 || N == 0) {
        if (dS && N) GNAN_CUDA(cudaMemsetAsync(dS, 0, sizeof(float) * N * C, st));
        if (dT && nT) GNAN_CUDA(cudaMemsetAsync(dT, 0, sizeof(float) * nT, st));
        return GNAN_OK;
    }
    AggArgs a{hop, R, N, ld_hop, T, table_per_row, nbins, Cr, rscale, S, C};
    const DsPlan p = plan_ds(R, N);
    const size_t need_ds = dS ? sizeof(float) * (size_t)p.nsb * N * C : 0;
    const size_t need_bs = Bsum ? 0 : sizeof(float) * (size_t)R * nbins * C;
    if (workspace_bytes < need_ds + need_bs || (!workspace && need_ds + need_bs)) {
        gnan_set_error("aggregate_rows_bwd: workspace %zu < %zu bytes", workspace_bytes, need_ds + need_bs);
        return GNAN_ERR_WORKSPACE;
    }
    float *dSpart = (float *)workspace;
    if (dT) {
        const float *bs = Bsum;
        if (!bs) {  // one extra pass to rebuild the bin sums; its `out` lands in the (not yet used) dS partial area
            float *tmp_bs = dSpart + (size_t)p.nsb * N * C;
            rc = gnan_agg_rows_fwd_cuda_cores(hop, R, N, ld_hop, T, table_per_row, nbins, Cr, rscale, S, C, dSpart, tmp_bs, stream);
            if (rc) return rc;
            bs = tmp_bs;
        }
        if (table_per_row) {
            agg_dt_per_row_kernel<<<(unsigned)ceil_div64(R * nbins, 256), 256, 0, st>>>(a, g, bs, dT);
        } else {
            GNAN_CUDA(cudaMemsetAsync(dT, 0, sizeof(float) * nT, st));
            const int nslab = (int)std::min<int64_t>(R, 4 * gnan_sm_count());
            agg_dt_global_kernel<<<nslab, 256, 0, st>>>(a, g, bs, ceil_div64(R, nslab), dT);
        }
        GNAN_LAUNCH_OK();
    }
    if (dS) {
        const int CC = C >= 4 ? 4 : (C >= 2 ? 2 : 1);
        dim3 grid((unsigned)p.ncol, (unsigned)p.nsb, (unsigned)((C + CC - 1) / CC));
        const size_t smem = sizeof(float) * CC * DS_RB * nbins;
        float *dst = p.nsb > 1 ? dSpart : dS;
        if (CC == 4) agg_rows_ds_kernel<4><<<grid, DS_THREADS, smem, st>>>(a, g, p.rows_per_sb, dst);
        else if (CC == 2) agg_rows_ds_kernel<2><<<grid, DS_THREADS, smem, st>>>(a, g, p.rows_per_sb, dst);
        else agg_rows_ds_kernel<1><<<grid, DS_THREADS, smem, st>>>(a, g, p.rows_per_sb, dst);
        GNAN_LAUNCH_OK();
        if (p.nsb > 1) {
            const size_t n = (size_t)N * C;
            rc = gnan_reduce_chunks(dSpart, p.nsb, n, n, dS, st);
            if (rc) return rc;
        }
    }
    return GNAN_OK;
}

static int check_bd(const char *who, const uint8_t *hop, const int64_t *hop_off, const int32_t *node_off, int B, const float *T,
                    int nbins, int Cr, const float *S, int C)
{
    GNAN_REQUIRE(B >= 0, "%s: negative batch", who);
    GNAN_REQUIRE(B == 0 || (hop && hop_off && node_off && T && S), "%s: NULL pointer", who);
    GNAN_REQUIRE(nbins >= 2 && nbins <= 256, "%s: nbins %d out of [2,256]", who, nbins);
    GNAN_REQUIRE(C >= 1 && (Cr == 1 || Cr == C), "%s: Cr must be 1 or C (Cr=%d C=%d)", who, Cr, C);
    return GNAN_OK;
}

extern "C" int gnan_aggregate_blockdiag_fwd(const uint8_t *hop, const int64_t *hop_off, const int32_t *node_off, int32_t B,
                                            const float *T, int table_per_row, int32_t nbins, int32_t Cr,
                                            const float *rscale, const float *S, int32_t C, int reduce_graph, float *out,
                                            gnan_stream_t stream)
{
    int rc = check_bd("aggregate_blockdiag_fwd", hop, hop_off, node_off, B, T, nbins, Cr, S, C);
    if (rc) return rc;
    if (B == 0) return GNAN_OK;
    GNAN_REQUIRE(out != nullptr, "aggregate_blockdiag_fwd: NULL out");
    BdArgs a{hop, hop_off, node_off, B, T, table_per_row, nbins, Cr, rscale, S, C, reduce_graph};
    const int blocks = (int)std::min<int64_t>(ceil_div64(B, 8), 8 * gnan_sm_count());
    const size_t smem = table_per_row ? 0 : sizeof(float) * (size_t)nbins * Cr;
    if (smem <= 48 * 1024) {
        if (C >= 4) agg_blockdiag_fwd_rows_kernel<4><<<blocks, 256, smem, (cudaStream_t)stream>>>(a, out);
        else if (C >= 2) agg_blockdiag_fwd_rows_kernel<2><<<blocks, 256, smem, (cudaStream_t)stream>>>(a, out);
        else agg_blockdiag_fwd_rows_kernel<1><<<blocks, 256, smem, (cudaStream_t)stream>>>(a, out);
    } else {
        agg_blockdiag_fwd_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(a, out);
    }
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}

extern "C" int gnan_aggregate_blockdiag_bwd(const uint8_t *hop, const int64_t *hop_off, const int32_t *node_off, int32_t B,
                                            const float *T, int table_per_row, int32_t nbins, int32_t Cr,
                                            const float *rscale, const float *S, int32_t C, int reduce_graph,
                                            const float *g, float *dS, float *dT, gnan_stream_t stream)
{
    int rc = check_bd("aggregate_blockdiag_bwd", hop, hop_off, node_off, B, T, nbins, Cr, S, C);
    if (rc) return rc;
    if (B == 0) return GNAN_OK;
    GNAN_REQUIRE(g && dS && dT, "aggregate_blockdiag_bwd: NULL g/dS/dT");
    cudaStream_t st = (cudaStream_t)stream;
    BdArgs a{hop, hop_off, node_off, B, T, table_per_row, nbins, Cr, rscale, S, C, reduce_graph};
    if (!table_per_row) GNAN_CUDA(cudaMemsetAsync(dT, 0, sizeof(float) * nbins * Cr, st));
    const int blocks = (int)std::min<int64_t>(ceil_div64(B, 8), 4 * gnan_sm_count());
    const size_t smem_g = sizeof(float) * (size_t)nbins * Cr * (1 + 8 * 32);
    if (!table_per_row && smem_g <= 200 * 1024) {       // global table: lane-private accumulators, one pass
        GNAN_CUDA(cudaFuncSetAttribute(agg_blockdiag_bwd_global_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_g));
        agg_blockdiag_bwd_global_kernel<<<blocks, 256, smem_g, st>>>(a, g, dS, dT);
        GNAN_LAUNCH_OK();
        return GNAN_OK;
    }
    const size_t smem = sizeof(float) * (size_t)nbins * Cr * (table_per_row ? 8 : 1);
    agg_blockdiag_bwd_kernel<<<blocks, 256, smem, st>>>(a, g, dS, dT);
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}
