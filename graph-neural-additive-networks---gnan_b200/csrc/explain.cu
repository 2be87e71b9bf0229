// Per-prediction attributions (gnan_b200.interpret.explain): the contribution of every shape function k to an output row,
//   F[r,k,c] = sum_j W[r,j,c'] f_k(x_jk)[c]                         (node rows: the reference's mf, GNAN.py:68-70)
//   F[b,k,c] = sum_{i in b} sum_j W[i,j,c'] f_k(x_jk)[c]            (graph rows: mf.sum(dim=1))
// computed on the compressed feature form of gnan_b200/sparse.py (per feature a baseline entry + exceptions sorted by row), so
// that the work is (rows) x (exceptions), never rows x N x K:
//   F[r,k,c] = Y[base_k,c] * sum_j W[r,j,c'] + sum_{e in seg(k, graph(r))} W[r,row(e),c'] * (Y[e,c] - Y[base_k,c]).
// Deterministic: every output element is one fixed-order sum written once, no atomics on floats.
#include <algorithm>

#include "common.cuh"

namespace {

// seg[k*(B+1)+b] = first exception of feature k whose row is >= node_off[b] (lower bound inside the feature's sorted exceptions)
__global__ void explain_segments_kernel(const int64_t *__restrict__ grp_ptr, const int64_t *__restrict__ ent_row, int K,
                                        const int32_t *__restrict__ node_off, int B, int64_t *__restrict__ seg)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)K * (B + 1)) return;
    const int k = (int)(t / (B + 1)), b = (int)(t % (B + 1));
    const int64_t key = node_off[b];
    int64_t lo = grp_ptr[k] + 1, hi = grp_ptr[k + 1];
    while (lo < hi) {
        const int64_t mid = lo + (hi - lo) / 2;
        if (ent_row[mid] < key) lo = mid + 1; else hi = mid;
    }
    seg[t] = lo;
}

// one thread per (graph, feature, channel): a fixed-order walk over the feature's exceptions inside the graph
__global__ void explain_graph_kernel(const float *__restrict__ Y, const int64_t *__restrict__ grp_ptr, const int64_t *__restrict__ ent_row,
                                     const int64_t *__restrict__ seg, int K, int B, int C, const float *__restrict__ colw,
                                     const float *__restrict__ colw_sum, float *__restrict__ F)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)B * K * C) return;
    const int c = (int)(t % C);
    const int64_t bk = t / C;
    const int k = (int)(bk % K), b = (int)(bk / K);
    const int64_t s0 = seg[(int64_t)k * (B + 1) + b], s1 = seg[(int64_t)k * (B + 1) + b + 1];
    const float yb = Y[grp_ptr[k] * C + c];
    float acc = 0.f;
    for (int64_t e = s0; e < s1; ++e) acc += colw[ent_row[e] * C + c] * (Y[e * C + c] - yb);
    F[t] = yb * colw_sum[(int64_t)b * C + c] + acc;
}

constexpr int ROWS_THREADS = 256;
constexpr int ROWS_MAX_RB = 32;      // rows of one CTA: one lane per row

struct RowsArgs {
    const uint8_t *hop;
    int64_t ld_hop;
    const int64_t *hop_off;          // NULL: dense row block (B == 1)
    const int32_t *node_off;
    int B;
    int64_t ncols;                   // columns staged per row: N (dense) / largest graph (packed)
    const int64_t *rows;             // output row -> hop row / global node, or NULL
    int64_t R;
    const float *T;
    int table_per_row, nbins, Cr;
    const float *rscale;
    const float *Y;
    const int64_t *grp_ptr, *ent_row, *seg;
    int K, C;
    float *F;
    int rb;                          // rows per CTA
    int lds;                         // staged bytes per row
};

// Node rows. A CTA owns `rb` output rows: it stages their hop rows in shared memory (coalesced byte loads), builds each row's
// weights w_r[d,c] = T[t_r,d,c'] * rscale[r,d] and bin histogram (rowW[r,c] = sum_d w_r[d,c] cnt_r[d]), then its warps take the
// features in turn; lane l holds row l and walks the feature's exception segment of its row's graph (the same segment for every
// lane of a dense block: the exception's row and value are warp-broadcast loads). CC channels per walk.
template <int CC>
__global__ void __launch_bounds__(ROWS_THREADS) explain_rows_kernel(const RowsArgs a)
{
    // widest element type first: every array starts aligned to its own size, whatever rb, nbins and C are
    extern __shared__ __align__(16) unsigned char smem[];
    const int rb = a.rb, nb = a.nbins, C = a.C;
    int64_t *src_s = reinterpret_cast<int64_t *>(smem);                       // [rb] hop row / node
    int64_t *base_s = src_s + ROWS_MAX_RB;                                    // [rb] first hop byte of the row
    int64_t *col0_s = base_s + ROWS_MAX_RB;                                   // [rb] first node of the row's graph
    int *g_s = reinterpret_cast<int *>(col0_s + ROWS_MAX_RB);                 // [rb] graph of the row
    int *n_s = g_s + ROWS_MAX_RB;                                             // [rb] columns of the row (-1: no row)
    float *w_s = reinterpret_cast<float *>(n_s + ROWS_MAX_RB);                // [rb][nbins][C]
    float *roww_s = w_s + (size_t)rb * nb * C;                                // [rb][C]
    int *hist_s = reinterpret_cast<int *>(roww_s + (size_t)rb * C);            // [rb][nbins]
    uint8_t *hop_s = reinterpret_cast<uint8_t *>(hist_s + (size_t)rb * nb);   // [rb][lds]

    const int tid = threadIdx.x;
    const int64_t r0 = (int64_t)blockIdx.x * rb;
    if (tid < rb) {
        const int64_t r = r0 + tid;
        int n = -1, g = 0;
        int64_t src = 0, base = 0, col0 = 0;
        if (r < a.R) {
            src = a.rows ? a.rows[r] : r;
            if (a.hop_off) {
                int lo = 0, hi = a.B;                                         // last graph with node_off[g] <= src
                while (hi - lo > 1) {
                    const int mid = (lo + hi) >> 1;
                    if (a.node_off[mid] <= src) lo = mid; else hi = mid;
                }
                g = lo;
                col0 = a.node_off[g];
                n = a.node_off[g + 1] - a.node_off[g];
                base = a.hop_off[g] + (src - col0) * n;
            } else {
                n = (int)a.ncols;
                base = src * a.ld_hop;
            }
        }
        src_s[tid] = src; base_s[tid] = base; col0_s[tid] = col0; g_s[tid] = g; n_s[tid] = n;
    }
    for (int i = tid; i < rb * nb; i += ROWS_THREADS) hist_s[i] = 0;
    __syncthreads();
    for (int q = 0; q < rb; ++q) {
        const int n = n_s[q];
        const uint8_t *h = a.hop + base_s[q];
        for (int j = tid; j < n; j += ROWS_THREADS) {
            const uint8_t v = h[j];
            hop_s[(size_t)q * a.lds + j] = v;
            atomicAdd(&hist_s[q * nb + min((int)v, nb - 1)], 1);               // integer counts: order-independent
        }
    }
    for (int i = tid; i < rb * nb * C; i += ROWS_THREADS) {
        const int q = i / (nb * C), d = (i / C) % nb, c = i % C;
        float w = 0.f;
        if (n_s[q] >= 0) {
            const int64_t src = src_s[q];
            w = a.T[(a.table_per_row ? src * nb * a.Cr : 0) + (int64_t)d * a.Cr + (a.Cr == 1 ? 0 : c)];
            if (a.rscale) w *= a.rscale[src * nb + d];
        }
        w_s[i] = w;
    }
    __syncthreads();
    for (int i = tid; i < rb * C; i += ROWS_THREADS) {
        const int q = i / C, c = i % C;
        float s = 0.f;
        for (int d = 0; d < nb; ++d) s += w_s[((size_t)q * nb + d) * C + c] * (float)hist_s[q * nb + d];
        roww_s[i] = s;
    }
    __syncthreads();

    const int warp = tid >> 5, lane = tid & 31;
    if (lane >= rb || n_s[lane] < 0) return;                                  // no more barriers below
    const int g = g_s[lane];
    const int64_t col0 = col0_s[lane], r = r0 + lane;
    const uint8_t *hrow = hop_s + (size_t)lane * a.lds;
    const float *wrow = w_s + (size_t)lane * nb * C;
    float *Fr = a.F + r * a.K * C;
    for (int k = warp; k < a.K; k += ROWS_THREADS / 32) {
        const int64_t s0 = a.seg[(int64_t)k * (a.B + 1) + g], s1 = a.seg[(int64_t)k * (a.B + 1) + g + 1];
        const float *yb = a.Y + a.grp_ptr[k] * C;
        for (int c0 = 0; c0 < C; c0 += CC) {
            float acc[CC];
#pragma unroll
            for (int u = 0; u < CC; ++u) acc[u] = 0.f;
            for (int64_t e = s0; e < s1; ++e) {
                const int d = min((int)hrow[a.ent_row[e] - col0], nb - 1);
                const float *ye = a.Y + e * C;
                const float *wd = wrow + d * C;
#pragma unroll
                for (int u = 0; u < CC; ++u)
                    if (c0 + u < C) acc[u] += wd[c0 + u] * (ye[c0 + u] - yb[c0 + u]);
            }
#pragma unroll
            for (int u = 0; u < CC; ++u)
                if (c0 + u < C) Fr[k * C + c0 + u] = yb[c0 + u] * roww_s[lane * C + c0 + u] + acc[u];
        }
    }
}

// the layout of explain_rows_kernel: row metadata, weights, row sums, histograms, hop bytes
size_t rows_smem_bytes(int rb, int nbins, int C, int lds)
{
    return ROWS_MAX_RB * (3 * 8 + 2 * 4) + ((size_t)rb * nbins * C + (size_t)rb * C + (size_t)rb * nbins) * 4 + (size_t)rb * lds;
}

constexpr size_t ROWS_SMEM_MAX = 200 * 1024;

}  // namespace

extern "C" int gnan_explain_segments(const int64_t *grp_ptr, const int64_t *ent_row, int32_t K, const int32_t *node_off, int32_t B,
                                     int64_t *seg, gnan_stream_t stream)
{
    GNAN_REQUIRE(K >= 1 && B >= 0, "explain_segments: bad sizes");
    GNAN_REQUIRE(grp_ptr && ent_row && node_off && seg, "explain_segments: NULL pointer");
    const int64_t n = (int64_t)K * (B + 1);
    explain_segments_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, (cudaStream_t)stream>>>(grp_ptr, ent_row, K, node_off, B, seg);
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}

extern "C" int gnan_explain_graph_features(const float *Y, const int64_t *grp_ptr, const int64_t *ent_row, const int64_t *seg, int32_t K,
                                           int32_t B, int32_t C, const float *colw, const float *colw_sum, float *F, gnan_stream_t stream)
{
    GNAN_REQUIRE(K >= 1 && B >= 0 && C >= 1, "explain_graph_features: bad sizes");
    if (B == 0) return GNAN_OK;
    GNAN_REQUIRE(Y && grp_ptr && ent_row && seg && colw && colw_sum && F, "explain_graph_features: NULL pointer");
    const int64_t n = (int64_t)B * K * C;
    explain_graph_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, (cudaStream_t)stream>>>(Y, grp_ptr, ent_row, seg, K, B, C, colw, colw_sum, F);
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}

extern "C" int gnan_explain_rows_features(const uint8_t *hop, int64_t ld_hop, const int64_t *hop_off, const int32_t *node_off, int32_t B,
                                          int64_t ncols, const int64_t *rows, int64_t R, const float *T, int table_per_row, int32_t nbins,
                                          int32_t Cr, const float *rscale, const float *Y, const int64_t *grp_ptr, const int64_t *ent_row,
                                          const int64_t *seg, int32_t K, int32_t C, float *F, gnan_stream_t stream)
{
    GNAN_REQUIRE(R >= 0 && B >= 1 && K >= 1 && C >= 1 && ncols >= 0 && nbins >= 1 && nbins <= 256 && (Cr == 1 || Cr == C),
                 "explain_rows_features: bad sizes");
    GNAN_REQUIRE(hop_off || (B == 1 && ld_hop >= ncols), "explain_rows_features: a dense row block has B == 1 and ld_hop >= ncols");
    if (R == 0) return GNAN_OK;
    GNAN_REQUIRE(hop && node_off && T && Y && grp_ptr && ent_row && seg && F, "explain_rows_features: NULL pointer");
    int lds = (int)((ncols + 3) / 4 * 4);
    if (((lds / 4) & 1) == 0) lds += 4;          // odd word stride: lanes (rows) reading the same column hit distinct banks
    int rb = ROWS_MAX_RB;
    while (rb > 1 && rows_smem_bytes(rb, nbins, C, lds) > ROWS_SMEM_MAX) rb >>= 1;
    const size_t smem = rows_smem_bytes(rb, nbins, C, lds);
    if (smem > ROWS_SMEM_MAX) {
        gnan_set_error("explain_rows_features: a row of %lld columns, %d bins and %d channels does not fit shared memory", (long long)ncols, nbins, C);
        return GNAN_ERR_UNSUPPORTED;
    }
    RowsArgs a{hop, ld_hop, hop_off, node_off, B, ncols, rows, R, T, table_per_row, nbins, Cr, rscale, Y, grp_ptr, ent_row, seg, K, C, F, rb, lds};
    const unsigned grid = (unsigned)ceil_div64(R, rb);
    cudaStream_t st = (cudaStream_t)stream;
#define GNAN_EXPLAIN_ROWS(CC)                                                                                                  \
    do {                                                                                                                       \
        GNAN_CUDA(cudaFuncSetAttribute(explain_rows_kernel<CC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));     \
        explain_rows_kernel<CC><<<grid, ROWS_THREADS, smem, st>>>(a);                                                          \
    } while (0)
    if (C == 1) GNAN_EXPLAIN_ROWS(1);
    else if (C == 2) GNAN_EXPLAIN_ROWS(2);
    else if (C <= 4) GNAN_EXPLAIN_ROWS(4);
    else GNAN_EXPLAIN_ROWS(8);
#undef GNAN_EXPLAIN_ROWS
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}
