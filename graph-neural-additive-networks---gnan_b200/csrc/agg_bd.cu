// Block-diagonal aggregation with a per-graph readout (graph-level tasks on batches of small graphs): ONE pass over the hop
// bytes serves the forward and the whole backward.
//
// Reference lines replaced: models.py:366-384 / GNAN.py:64-79 with is_graph_task (rho on the n*n pairs of every graph, matmul,
// the two sums), batched_pyg_main.py:154-181 (same on the dense (sum N)^2 collate), and autograd through them.
//
// For a GLOBAL distance table T[d,c'] (c' = 1 or C channels) and an optional per-row normaliser r[i,d] (models.py:368-370):
//     out[b,c] = sum_{i,j in graph b} T[d_ij,c'] r[i,d_ij] S[j,c],      d_ij = min(hop[i,j], nbins-1)
// is bilinear in (T, S) once the pair statistics
//     P[j,d] = sum_{i: d_ij = d} r[i,d]                                  (per hop COLUMN j; channel independent)
// are known:  colw[j,c'] = sum_d T[d,c'] P[j,d]   and   Q[b,d,c] = sum_{j in b} S[j,c] P[j,d]   give
//     out[b,c] = sum_d T[d,c'] Q[b,d,c] = sum_j colw[j,c'] S[j,c],   dS[j,c] = g[b,c] colw[j,c'],   dT[d,c'] = sum_{b,c} g[b,c] Q[b,d,c].
// The forward kernel makes the only pass over the pairs (a warp per graph, a lane per hop column, P in lane-private shared
// memory bins: no atomics, no cross-lane traffic in the pair loop) and saves colw [sumN,Cr] and Q [B,nbins,C]; the backward
// is two small streaming kernels that never touch the hop bytes. Everything is deterministic (fixed summation orders).
#include <algorithm>

#include "common.cuh"

namespace {

constexpr int BDG_RB = 8;            // hop rows per staged block of the normaliser table
constexpr int BDG_WARPS = 8;
constexpr int BDG_MAX_NBINS = 64;    // two bins per lane in the Q reduction
constexpr int BDG_SLABS = 1024;      // graph slabs of the dT reduction (at most; >= 8 graphs per slab)

struct BdgArgs {
    const uint8_t *hop;
    const int64_t *hop_off;
    const int32_t *node_off;
    int B;
    const float *T;
    int nbins, Cr;
    const float *rscale;
    const float *S;
    int C;
    float *out, *colw, *Q;
    int32_t *next;      // work counter (graphs are handed out dynamically: their cost varies like n^2)
};

__device__ __forceinline__ float lds_f32(uint32_t a)
{
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts_f32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" :: "r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void sts_v4(uint32_t a, float4 v)
{
    asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" :: "r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// VEC: the normaliser rows are staged with 16-byte loads (nbins % 4 == 0), else element by element.
// The pair loop is branch free: rows past the end of the graph read zero normaliser rows, columns past the end add 0, and
// the hop bytes + normaliser rows of row block k+1 are in flight (registers) while block k updates the bins.
template <int CC, bool VEC>
__global__ void __launch_bounds__(BDG_WARPS * 32)
agg_bd_graph_fwd_kernel(BdgArgs a)
{
    extern __shared__ __align__(16) float bdg_sm[];
    constexpr int NPF = VEC ? BDG_RB * BDG_MAX_NBINS / 128 : BDG_RB * BDG_MAX_NBINS / 32;     // prefetch registers (float4 / float)
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int nb = a.nbins, nb1 = nb - 1;
    const int nT = nb * a.Cr, nT4 = (nT + 3) & ~3;
    float *sT = bdg_sm;                                               // [nbins*Cr] table copy, CTA wide
    float *P = bdg_sm + nT4 + (size_t)w * (nb * 32 + BDG_RB * nb);    // [nbins][32] lane-private bins of this warp
    float *rs = P + nb * 32;                                          // [RB][nbins] normaliser rows of the current row block
    const uint32_t Pa = (uint32_t)__cvta_generic_to_shared(P) + 4u * lane, rsa = (uint32_t)__cvta_generic_to_shared(rs);
    for (int t = threadIdx.x; t < nT; t += blockDim.x) sT[t] = a.T[t];
    for (int d = 0; d < nb; ++d) P[d * 32 + lane] = 0.f;
    __syncthreads();
    const int rsn = BDG_RB * nb;                                      // floats per staged block
    for (;;) {
        int b = 0;
        if (lane == 0) b = atomicAdd(a.next, 1);
        b = __shfl_sync(0xffffffffu, b, 0);
        if (b >= a.B) break;
        const int n0 = a.node_off[b], n = a.node_off[b + 1] - n0;
        const uint8_t *hb = a.hop + a.hop_off[b];
        const float *rg = a.rscale ? a.rscale + (int64_t)n0 * nb : nullptr;
        const int rtot = n * nb;
        float q0[CC], q1[CC];
#pragma unroll
        for (int c = 0; c < CC; ++c) q0[c] = q1[c] = 0.f;
        for (int jq = 0; jq < n; jq += 32) {
            const int j = jq + lane;
            const bool jv = j < n;
            const uint8_t *hp = hb + (jv ? j : 0);                   // hop column of this lane (column 0 when past the end)
            float sown[CC];
#pragma unroll
            for (int c = 0; c < CC; ++c) sown[c] = (jv && c < a.C) ? a.S[(int64_t)(n0 + j) * a.C + c] : 0.f;
            int dmax = 0;
            // two register sets (A, B) of hop bytes + normaliser rows: block k+1 loads while block k updates the bins
            int hA[BDG_RB], hB[BDG_RB];
            float4 rA4[VEC ? NPF : 1], rB4[VEC ? NPF : 1];
            float rA1[VEC ? 1 : NPF], rB1[VEC ? 1 : NPF];
            const int nm1 = n - 1;
            auto load = [&](int i0, int (&h)[BDG_RB], float4 (&r4)[VEC ? NPF : 1], float (&r1)[VEC ? 1 : NPF]) {
#pragma unroll
                for (int u = 0; u < BDG_RB; ++u) h[u] = (int)hp[(uint32_t)(min(i0 + u, nm1) * n)];   // rows past the end: any row (they add 0)
                if (rg) {
                    const int left = rtot - i0 * nb;                  // floats of the normaliser left from this block on
                    const float *src = rg + i0 * nb;
                    if (VEC) {
#pragma unroll
                        for (int k = 0; k < NPF; ++k) {
                            const int e = lane * 4 + 128 * k;
                            r4[k] = (e < rsn && e < left) ? *reinterpret_cast<const float4 *>(src + e) : make_float4(0.f, 0.f, 0.f, 0.f);
                        }
                    } else {
#pragma unroll
                        for (int k = 0; k < NPF; ++k) {
                            const int e = lane + 32 * k;
                            r1[k] = (e < rsn && e < left) ? src[e] : 0.f;
                        }
                    }
                }
            };
            auto work = [&](int i0, const int (&h)[BDG_RB], const float4 (&r4)[VEC ? NPF : 1], const float (&r1)[VEC ? 1 : NPF]) {
                if (rg) {
                    if (VEC) {
#pragma unroll
                        for (int k = 0; k < NPF; ++k)
                            if (lane * 4 + 128 * k < rsn) sts_v4(rsa + 16u * lane + 512u * k, r4[k]);
                    } else {
#pragma unroll
                        for (int k = 0; k < NPF; ++k)
                            if (lane + 32 * k < rsn) sts_f32(rsa + 4u * lane + 128u * k, r1[k]);
                    }
                    __syncwarp();
                }
                int d[BDG_RB];
                float v[BDG_RB];
#pragma unroll
                for (int u = 0; u < BDG_RB; ++u) {
                    d[u] = min(h[u], nb1);
                    dmax = max(dmax, d[u]);
                    // rows past the end read a zero normaliser row (or add 0 without a normaliser). Lanes past the last column
                    // walk column 0: their bins hold finite garbage that is multiplied by S = 0 / never written out.
                    v[u] = rg ? lds_f32(rsa + 4u * (uint32_t)(u * nb + d[u])) : (i0 + u < n ? 1.f : 0.f);
                }
                // bins are read-modify-written two rows at a time (both loads in flight; equal bins are chained in registers)
#pragma unroll
                for (int u = 0; u < BDG_RB; u += 2) {
                    const uint32_t pa0 = Pa + 128u * (uint32_t)d[u], pa1 = Pa + 128u * (uint32_t)d[u + 1];
                    const float p0 = lds_f32(pa0), p1 = lds_f32(pa1);
                    const float n0v = p0 + v[u];
                    const float n1v = (d[u + 1] == d[u] ? n0v : p1) + v[u + 1];
                    sts_f32(pa0, n0v);
                    sts_f32(pa1, n1v);
                }
                if (rg) __syncwarp();
            };
            load(0, hA, rA4, rA1);
            for (int i0 = 0; i0 < n; i0 += 2 * BDG_RB) {
                const bool second = i0 + BDG_RB < n;
                if (second) load(i0 + BDG_RB, hB, rB4, rB1);
                work(i0, hA, rA4, rA1);
                if (second) {
                    if (i0 + 2 * BDG_RB < n) load(i0 + 2 * BDG_RB, hA, rA4, rA1);
                    work(i0 + BDG_RB, hB, rB4, rB1);
                }
            }
            // bins above the deepest level seen in this column block are untouched (still zero)
            const int dm = __reduce_max_sync(0xffffffffu, dmax);
            // colw[j,c'] = sum_d T[d,c'] P[j,d]
            for (int cr = 0; cr < a.Cr; ++cr) {
                float acc = 0.f;
                for (int d = 0; d <= dm; ++d) acc = fmaf(sT[d * a.Cr + cr], P[d * 32 + lane], acc);
                if (jv) a.colw[(int64_t)(n0 + j) * a.Cr + cr] = acc;
            }
            // Q[b,d,c] += sum_j S[j,c] P[j,d]: lane t owns bins t and t+32 and walks the 32 columns in a rotated order
            // (bank (l + t) % 32: conflict free)
            const bool hi = dm >= 32;
            __syncwarp();
#pragma unroll 4
            for (int l = 0; l < 32; ++l) {
                const int jj = (l + lane) & 31;
                const float p0 = lane <= dm ? P[lane * 32 + jj] : 0.f;
                const float p1 = (hi && lane + 32 <= dm) ? P[(lane + 32) * 32 + jj] : 0.f;
#pragma unroll
                for (int c = 0; c < CC; ++c) {
                    const float s = __shfl_sync(0xffffffffu, sown[c], jj);      // S[jq + jj, c] (0 beyond the graph or C)
                    q0[c] = fmaf(p0, s, q0[c]);
                    q1[c] = fmaf(p1, s, q1[c]);
                }
            }
            __syncwarp();
            for (int d = 0; d <= dm; ++d) P[d * 32 + lane] = 0.f;    // ready for the next column block / graph
            __syncwarp();
        }
        // Q[b,:,:] (all bins: zeros included, no memset needed) and out[b,c] = sum_d T[d,c'] Q[b,d,c]
#pragma unroll
        for (int c = 0; c < CC; ++c) {
            if (c < a.C) {
                const int cr = a.Cr == 1 ? 0 : c;
                float o = 0.f;
                if (lane < nb) {
                    a.Q[((int64_t)b * nb + lane) * a.C + c] = q0[c];
                    o = sT[lane * a.Cr + cr] * q0[c];
                }
                if (lane + 32 < nb) {
                    a.Q[((int64_t)b * nb + lane + 32) * a.C + c] = q1[c];
                    o = fmaf(sT[(lane + 32) * a.Cr + cr], q1[c], o);
                }
#pragma unroll
                for (int s = 16; s > 0; s >>= 1) o += __shfl_xor_sync(0xffffffffu, o, s);
                if (lane == 0) a.out[(int64_t)b * a.C + c] = o;
            }
        }
    }
}

// dS[j,c] = g[b,c] * colw[j,c']: a warp per graph
__global__ void __launch_bounds__(256)
agg_bd_graph_ds_kernel(const int32_t *__restrict__ node_off, int B, int Cr, int C, const float *__restrict__ g,
                       const float *__restrict__ colw, float *__restrict__ dS)
{
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t b = warp; b < B; b += nwarps) {
        const int64_t n0 = node_off[b], n1 = node_off[b + 1];
        for (int64_t t = n0 * C + lane; t < n1 * C; t += 32) {
            const int64_t j = t / C;
            const int c = (int)(t - j * C);
            dS[t] = g[b * C + c] * colw[j * Cr + (Cr == 1 ? 0 : c)];
        }
    }
}

// partial[slab][d*C+c] = sum_{b in slab} g[b,c] Q[b,d,c]  (fixed order)
__global__ void __launch_bounds__(128)
agg_bd_graph_dt_partial_kernel(int B, int nbins, int C, const float *__restrict__ g, const float *__restrict__ Q,
                               float *__restrict__ partial)
{
    const int per = (B + gridDim.x - 1) / gridDim.x;
    const int b0 = blockIdx.x * per, b1 = min(B, b0 + per);
    const int ne = nbins * C;
    for (int e = threadIdx.x; e < ne; e += blockDim.x) {
        const int c = e % C;
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
        int b = b0;
        for (; b + 3 < b1; b += 4) {
            s0 = fmaf(g[(int64_t)b * C + c], Q[(int64_t)b * ne + e], s0);
            s1 = fmaf(g[(int64_t)(b + 1) * C + c], Q[(int64_t)(b + 1) * ne + e], s1);
            s2 = fmaf(g[(int64_t)(b + 2) * C + c], Q[(int64_t)(b + 2) * ne + e], s2);
            s3 = fmaf(g[(int64_t)(b + 3) * C + c], Q[(int64_t)(b + 3) * ne + e], s3);
        }
        for (; b < b1; ++b) s0 = fmaf(g[(int64_t)b * C + c], Q[(int64_t)b * ne + e], s0);
        partial[(int64_t)e * gridDim.x + blockIdx.x] = (s0 + s1) + (s2 + s3);      // [entry][slab]: the final sum reads it coalesced
    }
}

// dT[d,c'] = sum over slabs (and over c when the table has one channel) of the partial sums: a warp per table entry, lanes
// stride over the slabs, fixed shuffle tree
__global__ void __launch_bounds__(256)
agg_bd_graph_dt_final_kernel(int nslab, int nbins, int Cr, int C, const float *__restrict__ partial, float *__restrict__ dT)
{
    const int lane = threadIdx.x & 31;
    const int t = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (t >= nbins * Cr) return;
    const int d = t / Cr, cr = t % Cr;
    const int ne = nbins * C;
    float s = 0.f;
    (void)ne;
    for (int sl = lane; sl < nslab; sl += 32) {
        if (Cr == 1) {
            for (int c = 0; c < C; ++c) s += partial[(int64_t)(d * C + c) * nslab + sl];
        } else {
            s += partial[(int64_t)(d * C + cr) * nslab + sl];
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) dT[t] = s;
}

}  // namespace

extern "C" int gnan_aggregate_blockdiag_graph_supported(int32_t nbins, int32_t Cr, int32_t C)
{
    return nbins >= 2 && nbins <= BDG_MAX_NBINS && C >= 1 && C <= 4 && (Cr == 1 || Cr == C);
}

extern "C" int gnan_aggregate_blockdiag_graph_fwd(const uint8_t *hop, const int64_t *hop_off, const int32_t *node_off, int32_t B,
                                                  const float *T, int32_t nbins, int32_t Cr, const float *rscale, const float *S,
                                                  int32_t C, float *out, float *colw, float *Q, int32_t *work_counter,
                                                  gnan_stream_t stream)
{
    GNAN_REQUIRE(B >= 0, "aggregate_blockdiag_graph_fwd: negative batch");
    if (B == 0) return GNAN_OK;
    if (!gnan_aggregate_blockdiag_graph_supported(nbins, Cr, C)) {
        gnan_set_error("aggregate_blockdiag_graph_fwd: needs 2 <= nbins <= %d, C <= 4, Cr in {1,C} (nbins=%d Cr=%d C=%d)", BDG_MAX_NBINS,
                       nbins, Cr, C);
        return GNAN_ERR_UNSUPPORTED;
    }
    GNAN_REQUIRE(hop && hop_off && node_off && T && S && out && colw && Q && work_counter, "aggregate_blockdiag_graph_fwd: NULL pointer");
    GNAN_REQUIRE(!rscale || (nbins & 3) != 0 || ((uintptr_t)rscale & 15) == 0, "aggregate_blockdiag_graph_fwd: rscale must be 16-byte aligned");
    BdgArgs a{hop, hop_off, node_off, B, T, nbins, Cr, rscale, S, C, out, colw, Q, work_counter};
    const size_t smem = sizeof(float) * ((size_t)((nbins * Cr + 3) & ~3) + (size_t)BDG_WARPS * (nbins * 32 + BDG_RB * nbins));
    cudaStream_t st = (cudaStream_t)stream;
    GNAN_CUDA(cudaMemsetAsync(work_counter, 0, sizeof(int32_t), st));
    auto launch = [&](auto kernel) -> int {
        // attribute + occupancy are looked up once per (kernel, shared-memory size): the calls cost tens of microseconds of host time
        // (all instantiations share ONE function-pointer type, hence one copy of these statics: the kernel is part of the key)
        static thread_local size_t cached_smem = 0;
        static thread_local int cached_per_sm = 0;
        static thread_local const void *cached_kernel = nullptr;
        if (cached_kernel != (const void *)kernel || cached_smem != smem || cached_per_sm == 0) {
            GNAN_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            GNAN_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&cached_per_sm, kernel, BDG_WARPS * 32, smem));
            cached_smem = smem;
            cached_kernel = (const void *)kernel;
        }
        const int per_sm = cached_per_sm;
        const int blocks = (int)std::min<int64_t>(ceil_div64(B, BDG_WARPS), (int64_t)std::max(per_sm, 1) * gnan_sm_count());
        kernel<<<blocks, BDG_WARPS * 32, smem, st>>>(a);      // persistent: every resident warp pulls graphs until none is left
        GNAN_LAUNCH_OK();
        return GNAN_OK;
    };
    const bool vec = (nbins & 3) == 0;
    if (C == 1) return vec ? launch(agg_bd_graph_fwd_kernel<1, true>) : launch(agg_bd_graph_fwd_kernel<1, false>);
    if (C == 2) return vec ? launch(agg_bd_graph_fwd_kernel<2, true>) : launch(agg_bd_graph_fwd_kernel<2, false>);
    return vec ? launch(agg_bd_graph_fwd_kernel<4, true>) : launch(agg_bd_graph_fwd_kernel<4, false>);
}

extern "C" size_t gnan_aggregate_blockdiag_graph_bwd_workspace_bytes(int32_t nbins, int32_t C)
{
    return sizeof(float) * (size_t)BDG_SLABS * nbins * C;
}

extern "C" int gnan_aggregate_blockdiag_graph_bwd(const int32_t *node_off, int32_t B, int32_t nbins, int32_t Cr, int32_t C,
                                                  const float *g, const float *colw, const float *Q, float *dS, float *dT,
                                                  void *workspace, size_t workspace_bytes, gnan_stream_t stream)
{
    GNAN_REQUIRE(B >= 0 && nbins >= 2 && C >= 1 && (Cr == 1 || Cr == C), "aggregate_blockdiag_graph_bwd: bad sizes");
    GNAN_REQUIRE(dT != nullptr, "aggregate_blockdiag_graph_bwd: NULL dT");
    cudaStream_t st = (cudaStream_t)stream;
    if (B == 0) {
        GNAN_CUDA(cudaMemsetAsync(dT, 0, sizeof(float) * nbins * Cr, st));
        return GNAN_OK;
    }
    GNAN_REQUIRE(node_off && g && colw && Q && dS, "aggregate_blockdiag_graph_bwd: NULL pointer");
    const size_t need = gnan_aggregate_blockdiag_graph_bwd_workspace_bytes(nbins, C);
    if (!workspace || workspace_bytes < need) {
        gnan_set_error("aggregate_blockdiag_graph_bwd: workspace %zu < %zu bytes", workspace_bytes, need);
        return GNAN_ERR_WORKSPACE;
    }
    const int blocks = (int)std::min<int64_t>(ceil_div64(B, 8), 8 * gnan_sm_count());
    agg_bd_graph_ds_kernel<<<blocks, 256, 0, st>>>(node_off, B, Cr, C, g, colw, dS);
    GNAN_LAUNCH_OK();
    const int nslab = (int)std::max<int64_t>(1, std::min<int64_t>(BDG_SLABS, B / 8));
    float *partial = (float *)workspace;
    agg_bd_graph_dt_partial_kernel<<<nslab, 128, 0, st>>>(B, nbins, C, g, Q, partial);
    GNAN_LAUNCH_OK();
    agg_bd_graph_dt_final_kernel<<<(unsigned)ceil_div64((int64_t)nbins * Cr * 32, 256), 256, 0, st>>>(nslab, nbins, Cr, C, partial, dT);
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}
