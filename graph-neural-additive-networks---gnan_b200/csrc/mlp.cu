// Grouped scalar-input MLPs (the K shape functions f_k and the distance function rho), fp32 FFMA path.
//
// Reference lines replaced: GNAN.py:57-62 (K-iteration module loop + slice assignment), :157 (feature sum),
// models.py:360-365, batched_pyg_main.py:144-148; backward = autograd through the same (trainer.py:66).
//
// Design (see DESIGN.md "mlp"): a CTA owns a 128-row tile. Activations live in shared memory as
// [row][unit] with a +4 float pad (conflict-free 128-bit accesses); the hidden HxH layers are register-tiled
// SGEMMs (thread tile 8 rows x H/8 units, both operands read with LDS.128 along the contraction index).
// Layer 1 is an outer product generated straight into shared memory (x*w1+b1, ReLU); the last layer and the sum
// over groups are fused so the reference's [N,K,C] tensor never exists. Backward recomputes activations.
#include <algorithm>

#include "common.cuh"

namespace {

constexpr int TM = 128;  // rows per tile
constexpr int NT = 128;  // threads per CTA

struct MlpKArgs {
    const float *u;
    int64_t R, ldu;
    int G, C, nh;
    const float *w1, *b1, *wh, *bh, *wo, *bo;
    uint32_t drop_thresh;  // 0 = no dropout
    float drop_scale;
    uint64_t seed;
    const uint64_t *seed_dev;  // optional device-resident seed word, XORed into `seed` at kernel start (CUDA-graph replays)
    float *du;  // backward only: [R,G] gradient w.r.t. the inputs, or NULL
    // entries mode (gnan_mlp_entries_*): u is a flat value list grouped by feature, group g owns entries
    // [grp_ptr[g], grp_ptr[g+1]); rows of a group are its entries, outputs / dY are indexed by entry. NULL = dense mode.
    const int64_t *grp_ptr;
    const int32_t *items;  // forward, entries mode: [n_items][2] = (group, 128-entry tile of that group), one CTA each
};

__device__ __forceinline__ float relu(float v) { return v > 0.f ? v : 0.f; }

// ---- micro-kernels -------------------------------------------------------------------------------------------
// MK1: acc[e][f] += sum_k A[(e*16+ty)][k] * B[(f*8+tx)][k]      A:[128][lda]  B:[>=TN*8][ldb]   (dot form)
template <int TN>
__device__ __forceinline__ void mk1(const float *__restrict__ sA, int lda, const float *__restrict__ sB, int ldb, int K,
                                    int ty, int tx, float (&acc)[8][TN])
{
#pragma unroll 2
    for (int k = 0; k < K; k += 4) {
        float4 a[8], b[TN];
#pragma unroll
        for (int e = 0; e < 8; ++e) a[e] = *reinterpret_cast<const float4 *>(sA + (e * 16 + ty) * lda + k);
#pragma unroll
        for (int f = 0; f < TN; ++f) b[f] = *reinterpret_cast<const float4 *>(sB + (f * 8 + tx) * ldb + k);
#pragma unroll
        for (int e = 0; e < 8; ++e)
#pragma unroll
            for (int f = 0; f < TN; ++f) {
                acc[e][f] = fmaf(a[e].x, b[f].x, acc[e][f]);
                acc[e][f] = fmaf(a[e].y, b[f].y, acc[e][f]);
                acc[e][f] = fmaf(a[e].z, b[f].z, acc[e][f]);
                acc[e][f] = fmaf(a[e].w, b[f].w, acc[e][f]);
            }
    }
}

// MK2: acc[e][v*4+f] += sum_k A[(e*16+ty)][k] * B[k][v*32+tx*4+f]   A:[128][lda]  B:[K][ldb], n < Nn valid
template <int NV>
__device__ __forceinline__ void mk2(const float *__restrict__ sA, int lda, const float *__restrict__ sB, int ldb, int K,
                                    int Nn, int ty, int tx, float (&acc)[8][NV * 4])
{
    bool ok[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) ok[v] = (v * 32 + tx * 4) < Nn;
#pragma unroll 1
    for (int k = 0; k < K; k += 4) {
        float4 a[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) a[e] = *reinterpret_cast<const float4 *>(sA + (e * 16 + ty) * lda + k);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            float4 b[NV];
#pragma unroll
            for (int v = 0; v < NV; ++v)
                b[v] = ok[v] ? *reinterpret_cast<const float4 *>(sB + (k + kk) * ldb + v * 32 + tx * 4)
                             : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const float av = kk == 0 ? a[e].x : kk == 1 ? a[e].y : kk == 2 ? a[e].z : a[e].w;
#pragma unroll
                for (int v = 0; v < NV; ++v) {
                    acc[e][v * 4 + 0] = fmaf(av, b[v].x, acc[e][v * 4 + 0]);
                    acc[e][v * 4 + 1] = fmaf(av, b[v].y, acc[e][v * 4 + 1]);
                    acc[e][v * 4 + 2] = fmaf(av, b[v].z, acc[e][v * 4 + 2]);
                    acc[e][v * 4 + 3] = fmaf(av, b[v].w, acc[e][v * 4 + 3]);
                }
            }
        }
    }
}

// MK3: acc[e][f] += sum_{k<TM} A[k][ty2*8+e] * B[k][tx2*4+f]     A:[TM][lda] (m<M valid)  B:[TM][ldb] (n<Nn valid)
__device__ __forceinline__ void mk3(const float *__restrict__ sA, int lda, const float *__restrict__ sB, int ldb, int M,
                                    int Nn, int ty2, int tx2, float (&acc)[8][4])
{
    if (ty2 * 8 >= M || tx2 * 4 >= Nn) return;
#pragma unroll 4
    for (int k = 0; k < TM; ++k) {
        const float4 a0 = *reinterpret_cast<const float4 *>(sA + k * lda + ty2 * 8);
        const float4 a1 = *reinterpret_cast<const float4 *>(sA + k * lda + ty2 * 8 + 4);
        const float4 b = *reinterpret_cast<const float4 *>(sB + k * ldb + tx2 * 4);
        const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            acc[e][0] = fmaf(a[e], b.x, acc[e][0]);
            acc[e][1] = fmaf(a[e], b.y, acc[e][1]);
            acc[e][2] = fmaf(a[e], b.z, acc[e][2]);
            acc[e][3] = fmaf(a[e], b.w, acc[e][3]);
        }
    }
}

// copy an [rows][H] fp32 matrix (global, contiguous) into smem [rows][LD]
template <int H>
__device__ __forceinline__ void load_matrix(float *__restrict__ dst, const float *__restrict__ src, int rows, int tid)
{
    constexpr int LD = H + 4;
    constexpr int V = H / 4;
    for (int i = tid; i < rows * V; i += NT) {
        const int r = i / V, c = i % V;
        *reinterpret_cast<float4 *>(dst + r * LD + c * 4) = __ldg(reinterpret_cast<const float4 *>(src) + i);
    }
}

// layer 1 for row `tid`: a0[i] = relu(x*w1[i]+b1[i]) * dropout  -> sAct0[tid][.]
template <int H>
__device__ __forceinline__ void gen_layer1(float *__restrict__ sAct0, const float *__restrict__ sW1,
                                           const float *__restrict__ sB1, float x, int tid, const MlpKArgs &a, int g,
                                           int64_t row)
{
    constexpr int LD = H + 4;
#pragma unroll 4
    for (int i = 0; i < H; i += 4) {
        const float4 w = *reinterpret_cast<const float4 *>(sW1 + i);
        const float4 b = *reinterpret_cast<const float4 *>(sB1 + i);
        float4 v;
        v.x = relu(fmaf(x, w.x, b.x));
        v.y = relu(fmaf(x, w.y, b.y));
        v.z = relu(fmaf(x, w.z, b.z));
        v.w = relu(fmaf(x, w.w, b.w));
        if (a.drop_thresh) {
            const uint64_t key = (((uint64_t)g) * (uint64_t)a.R + (uint64_t)row) * H + i;  // layer 0
            v.x *= gnan_dropout_mul(a.seed, key + 0, a.drop_thresh, a.drop_scale);
            v.y *= gnan_dropout_mul(a.seed, key + 1, a.drop_thresh, a.drop_scale);
            v.z *= gnan_dropout_mul(a.seed, key + 2, a.drop_thresh, a.drop_scale);
            v.w *= gnan_dropout_mul(a.seed, key + 3, a.drop_thresh, a.drop_scale);
        }
        *reinterpret_cast<float4 *>(sAct0 + tid * LD + i) = v;
    }
}

__device__ __forceinline__ uint64_t drop_key(const MlpKArgs &a, int layer, int g, int64_t row, int H, int unit)
{
    return ((((uint64_t)layer * a.G + g) * (uint64_t)a.R + (uint64_t)row) * H) + unit;
}

// ---- forward -------------------------------------------------------------------------------------------------
// grid (row tiles, group chunks); Spart[chunk][R][C]
template <int H>
__global__ void __launch_bounds__(NT, (H <= 64 ? 3 : 1))
mlp_fwd_kernel(MlpKArgs a, int KC, float *__restrict__ Spart)
{
    constexpr int LD = H + 4;
    constexpr int TN = H / 8;
    extern __shared__ __align__(16) float smem[];
    const int CP = (a.C + 7) / 8 * 8;
    float *sAct = smem;                 // [TM][LD]
    float *sW = sAct + TM * LD;         // [H][LD]
    float *sWo = sW + H * LD;           // [CP][LD]
    float *sS = sWo + CP * LD;          // [TM][CP]
    float *sX = sS + TM * CP;           // [KC][TM]
    float *sW1 = sX + KC * TM;          // [H]
    float *sB1 = sW1 + H;               // [H]
    float *sBh = sB1 + H;               // [H]
    float *sBo = sBh + H;               // [CP]

    const int tid = threadIdx.x, tx = tid & 7, ty = tid >> 3;
    if (a.seed_dev) a.seed ^= *a.seed_dev;
    int64_t row0 = (int64_t)blockIdx.x * TM, nrow = a.R, ebase = 0;
    int g0 = blockIdx.y * KC;
    int ng = min(KC, a.G - g0);
    if (a.items) {                       // entries mode: this CTA = one (group, tile) item; its rows are the group's entries
        g0 = a.items[2 * blockIdx.x];
        row0 = (int64_t)a.items[2 * blockIdx.x + 1] * TM;
        ng = 1;
        ebase = a.grp_ptr[g0];
        nrow = a.grp_ptr[g0 + 1] - ebase;
    }

    for (int i = tid; i < ng * TM; i += NT) {
        const int r = i / ng, kk = i % ng;
        const int64_t row = row0 + r;
        sX[kk * TM + r] = row < nrow ? __ldg(a.items ? a.u + ebase + row : a.u + row * a.ldu + g0 + kk) : 0.f;
    }
    for (int i = tid; i < TM * CP; i += NT) sS[i] = 0.f;
    for (int i = tid; i < CP * LD; i += NT) sWo[i] = 0.f;
    __syncthreads();

    for (int kk = 0; kk < ng; ++kk) {
        const int g = g0 + kk;
        // stage this group's small vectors, output weights and first hidden matrix
        for (int i = tid; i < H; i += NT) {
            sW1[i] = __ldg(a.w1 + (size_t)g * H + i);
            sB1[i] = a.b1 ? __ldg(a.b1 + (size_t)g * H + i) : 0.f;
        }
        for (int i = tid; i < a.C * (H / 4); i += NT) {
            const int c = i / (H / 4), q = i % (H / 4);
            *reinterpret_cast<float4 *>(sWo + c * LD + q * 4) =
                __ldg(reinterpret_cast<const float4 *>(a.wo + ((size_t)g * a.C + c) * H) + q);
        }
        for (int i = tid; i < CP; i += NT) sBo[i] = (a.bo && i < a.C) ? __ldg(a.bo + (size_t)g * a.C + i) : 0.f;
        if (a.nh > 0) load_matrix<H>(sW, a.wh + (size_t)g * H * H, H, tid);
        __syncthreads();
        gen_layer1<H>(sAct, sW1, sB1, sX[kk * TM + tid], tid, a, g, row0 + tid);
        __syncthreads();

        for (int l = 0; l < a.nh; ++l) {
            if (l > 0) load_matrix<H>(sW, a.wh + ((size_t)l * a.G + g) * H * H, H, tid);
            for (int i = tid; i < H; i += NT) sBh[i] = a.bh ? __ldg(a.bh + ((size_t)l * a.G + g) * H + i) : 0.f;
            if (l > 0) __syncthreads();
            float acc[8][TN];
#pragma unroll
            for (int e = 0; e < 8; ++e)
#pragma unroll
                for (int f = 0; f < TN; ++f) acc[e][f] = 0.f;
            mk1<TN>(sAct, LD, sW, LD, H, ty, tx, acc);
            __syncthreads();  // all reads of sAct / sW done (sBh was written before the barrier inside gen or above)
#pragma unroll
            for (int e = 0; e < 8; ++e)
#pragma unroll
                for (int f = 0; f < TN; ++f) {
                    const int r = e * 16 + ty, j = f * 8 + tx;
                    float v = relu(acc[e][f] + sBh[j]);
                    if (a.drop_thresh)
                        v *= gnan_dropout_mul(a.seed, drop_key(a, l + 1, g, row0 + r, H, j), a.drop_thresh, a.drop_scale);
                    sAct[r * LD + j] = v;
                }
            __syncthreads();
        }
        // output layer + accumulation over groups: sS[r][c] += a_last[r][:] . wo[c][:] + bo[c]
        for (int e0 = 0; e0 < CP / 8; ++e0) {
            float acc1[8][1];
#pragma unroll
            for (int e = 0; e < 8; ++e) acc1[e][0] = 0.f;
            mk1<1>(sAct, LD, sWo + e0 * 8 * LD, LD, H, ty, tx, acc1);
            const int c = e0 * 8 + tx;
            if (c < a.C) {
                const float bo = sBo[c];
#pragma unroll
                for (int e = 0; e < 8; ++e) sS[(e * 16 + ty) * CP + c] += acc1[e][0] + bo;
            }
        }
        __syncthreads();  // sAct / sWo / small vectors are rewritten by the next group
    }
    float *out = a.items ? Spart + ebase * a.C : Spart + (size_t)blockIdx.y * a.R * a.C;
    for (int i = tid; i < TM * a.C; i += NT) {
        const int r = i / a.C, c = i % a.C;
        if (row0 + r < nrow) out[(row0 + r) * a.C + c] = sS[r * CP + c];
    }
}

// ---- backward ------------------------------------------------------------------------------------------------
struct MlpGradPtrs {
    float *w1, *b1, *wh, *bh, *wo, *bo;  // bases of chunk 0
    size_t chunk_stride;                 // floats between consecutive chunks (0 if single chunk)
};

template <int H, int NH>
__global__ void __launch_bounds__(NT, (H <= 64 && NH <= 1 ? 2 : 1))
mlp_bwd_kernel(MlpKArgs a, const float *__restrict__ dS, MlpGradPtrs gp, int64_t ntiles)
{
    constexpr int LD = H + 4;
    constexpr int TN = H / 8;
    constexpr int NV = (H + 31) / 32;
    constexpr int NHA = NH > 0 ? NH : 1;
    extern __shared__ __align__(16) float smem[];
    const int CP = (a.C + 7) / 8 * 8;  // padded channel count
    const int CG = CP + 4;             // row stride of sG
    float *sAct = smem;                       // [NH+1][TM][LD]
    float *sW = sAct + (NH + 1) * TM * LD;    // [H][LD]   current hidden matrix (row j, col i)
    float *sWo = sW + H * LD;                 // [CP][LD]  wo rows (c), zero padded
    float *sDWo = sWo + CP * LD;              // [CP][LD]  dwo accumulator
    float *sG = sDWo + CP * LD;               // [TM][CG]  dS tile
    float *sX = sG + TM * CG;                 // [TM]
    float *sW1 = sX + TM;                     // [H]
    float *sB1 = sW1 + H;                     // [H]
    float *sBh = sB1 + H;                     // [NHA][H]

    const int tid = threadIdx.x, tx = tid & 7, ty = tid >> 3, tx2 = tid & 15, ty2 = tid >> 4;
    const int g = blockIdx.y;
    if (a.seed_dev) a.seed ^= *a.seed_dev;
    const float dscale = a.drop_thresh ? a.drop_scale : 1.f;

    // group constants
    for (int i = tid; i < H; i += NT) {
        sW1[i] = __ldg(a.w1 + (size_t)g * H + i);
        sB1[i] = a.b1 ? __ldg(a.b1 + (size_t)g * H + i) : 0.f;
        for (int l = 0; l < NH; ++l) sBh[l * H + i] = a.bh ? __ldg(a.bh + ((size_t)l * a.G + g) * H + i) : 0.f;
    }
    for (int i = tid; i < CP * LD; i += NT) { sWo[i] = 0.f; sDWo[i] = 0.f; }
    __syncthreads();
    for (int i = tid; i < a.C * (H / 4); i += NT) {
        const int c = i / (H / 4), q = i % (H / 4);
        *reinterpret_cast<float4 *>(sWo + c * LD + q * 4) =
            __ldg(reinterpret_cast<const float4 *>(a.wo + ((size_t)g * a.C + c) * H) + q);
    }
    if (NH == 1) load_matrix<H>(sW, a.wh + (size_t)g * H * H, H, tid);

    float accW[NHA][8][4];  // dWh[l][ty2*8+e][tx2*4+f]
#pragma unroll
    for (int l = 0; l < NHA; ++l)
#pragma unroll
        for (int e = 0; e < 8; ++e)
#pragma unroll
            for (int f = 0; f < 4; ++f) accW[l][e][f] = 0.f;
    float pbh[NHA];  // dbh[l][tid]   (tid < H)
#pragma unroll
    for (int l = 0; l < NHA; ++l) pbh[l] = 0.f;
    float pw1 = 0.f, pb1 = 0.f;  // dw1[tid], db1[tid]
    float pbo = 0.f;             // dbo[tid]  (tid < C)

    int64_t nrow = a.R, ebase = 0;
    if (a.grp_ptr) {                     // entries mode: the rows of group g are its entries
        ebase = a.grp_ptr[g];
        nrow = a.grp_ptr[g + 1] - ebase;
        ntiles = (nrow + TM - 1) / TM;
        dS += ebase * a.C;
    }
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int64_t row0 = t * TM;
        __syncthreads();  // previous tile fully consumed
        {
            const int64_t row = row0 + tid;
            sX[tid] = row < nrow ? __ldg(a.grp_ptr ? a.u + ebase + row : a.u + row * a.ldu + g) : 0.f;
        }
        for (int i = tid; i < TM * CP; i += NT) {
            const int r = i / CP, c = i % CP;
            sG[r * CG + c] = (row0 + r < nrow && c < a.C) ? __ldg(dS + (row0 + r) * a.C + c) : 0.f;
        }
        __syncthreads();
        gen_layer1<H>(sAct, sW1, sB1, sX[tid], tid, a, g, row0 + tid);
        __syncthreads();
        // ---- recompute forward activations a_1..a_NH
#pragma unroll
        for (int l = 0; l < NH; ++l) {
            if (NH > 1) {
                load_matrix<H>(sW, a.wh + ((size_t)l * a.G + g) * H * H, H, tid);
                __syncthreads();
            }
            float acc[8][TN];
#pragma unroll
            for (int e = 0; e < 8; ++e)
#pragma unroll
                for (int f = 0; f < TN; ++f) acc[e][f] = 0.f;
            mk1<TN>(sAct + l * TM * LD, LD, sW, LD, H, ty, tx, acc);
            float *dst = sAct + (l + 1) * TM * LD;
#pragma unroll
            for (int e = 0; e < 8; ++e)
#pragma unroll
                for (int f = 0; f < TN; ++f) {
                    const int r = e * 16 + ty, j = f * 8 + tx;
                    float v = relu(acc[e][f] + sBh[l * H + j]);
                    if (a.drop_thresh)
                        v *= gnan_dropout_mul(a.seed, drop_key(a, l + 1, g, row0 + r, H, j), a.drop_thresh, a.drop_scale);
                    dst[r * LD + j] = v;
                }
            __syncthreads();
        }
        // ---- output layer backward
        float *aL = sAct + NH * TM * LD;
        if (tid < a.C) {
            float s = 0.f;
            for (int r = 0; r < TM; ++r) s += sG[r * CG + tid];
            pbo += s;
        }
        // dWo[c][j] += sum_r g[r][c] * aL[r][j] : thread = (row slice ty2 of 16 rows, 4 columns tx2*4..), 8 channels at a time
        if (tx2 * 4 < H) {
            for (int c0 = 0; c0 < CP; c0 += 8) {
                float w[8][4];
#pragma unroll
                for (int e = 0; e < 8; ++e)
#pragma unroll
                    for (int f = 0; f < 4; ++f) w[e][f] = 0.f;
#pragma unroll 4
                for (int rr = 0; rr < 16; ++rr) {
                    const int r = ty2 * 16 + rr;
                    const float4 b = *reinterpret_cast<const float4 *>(aL + r * LD + tx2 * 4);
                    const float4 g0 = *reinterpret_cast<const float4 *>(sG + r * CG + c0);
                    const float4 g1 = *reinterpret_cast<const float4 *>(sG + r * CG + c0 + 4);
                    const float gv[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        w[e][0] = fmaf(gv[e], b.x, w[e][0]);
                        w[e][1] = fmaf(gv[e], b.y, w[e][1]);
                        w[e][2] = fmaf(gv[e], b.z, w[e][2]);
                        w[e][3] = fmaf(gv[e], b.w, w[e][3]);
                    }
                }
#pragma unroll
                for (int e = 0; e < 8; ++e)
                    if (c0 + e < a.C) {
#pragma unroll
                        for (int f = 0; f < 4; ++f) atomicAdd(sDWo + (c0 + e) * LD + tx2 * 4 + f, w[e][f]);
                    }
            }
        }
        // d = G . Wo   (K = CP), then dz = d * 1[aL>0] * dropout scale
        float d[8][NV * 4];
#pragma unroll
        for (int e = 0; e < 8; ++e)
#pragma unroll
            for (int f = 0; f < NV * 4; ++f) d[e][f] = 0.f;
        mk2<NV>(sG, CG, sWo, LD, CP, H, ty, tx, d);
#pragma unroll
        for (int e = 0; e < 8; ++e)
#pragma unroll
            for (int v = 0; v < NV; ++v)
#pragma unroll
                for (int f = 0; f < 4; ++f) {
                    const int r = e * 16 + ty, j = v * 32 + tx * 4 + f;
                    if (j < H) d[e][v * 4 + f] = aL[r * LD + j] > 0.f ? d[e][v * 4 + f] * dscale : 0.f;
                }
        __syncthreads();  // all reads of aL (dWo pass, masks) done
#pragma unroll
        for (int e = 0; e < 8; ++e)
#pragma unroll
            for (int v = 0; v < NV; ++v) {
                const int r = e * 16 + ty, j = v * 32 + tx * 4;
                if (j < H)
                    *reinterpret_cast<float4 *>(aL + r * LD + j) =
                        make_float4(d[e][v * 4 + 0], d[e][v * 4 + 1], d[e][v * 4 + 2], d[e][v * 4 + 3]);
            }
        __syncthreads();
        // ---- hidden layers, top down. sD = sAct[l+1] now holds dz_{l+1}
#pragma unroll
        for (int l = NH - 1; l >= 0; --l) {
            const float *sD = sAct + (l + 1) * TM * LD;
            float *aPrev = sAct + l * TM * LD;
            if (NH > 1) {
                load_matrix<H>(sW, a.wh + ((size_t)l * a.G + g) * H * H, H, tid);
                __syncthreads();
            }
            mk3(sD, LD, aPrev, LD, H, H, ty2, tx2, accW[l]);
            if (tid < H) {
                float s = 0.f;
                for (int r = 0; r < TM; ++r) s += sD[r * LD + tid];
                pbh[l] += s;
            }
#pragma unroll
            for (int e = 0; e < 8; ++e)
#pragma unroll
                for (int f = 0; f < NV * 4; ++f) d[e][f] = 0.f;
            mk2<NV>(sD, LD, sW, LD, H, H, ty, tx, d);
#pragma unroll
            for (int e = 0; e < 8; ++e)
#pragma unroll
                for (int v = 0; v < NV; ++v)
#pragma unroll
                    for (int f = 0; f < 4; ++f) {
                        const int r = e * 16 + ty, i = v * 32 + tx * 4 + f;
                        if (i < H) d[e][v * 4 + f] = aPrev[r * LD + i] > 0.f ? d[e][v * 4 + f] * dscale : 0.f;
                    }
            __syncthreads();  // mk3 / masks done reading aPrev, mk2 done reading sD
#pragma unroll
            for (int e = 0; e < 8; ++e)
#pragma unroll
                for (int v = 0; v < NV; ++v) {
                    const int r = e * 16 + ty, i = v * 32 + tx * 4;
                    if (i < H)
                        *reinterpret_cast<float4 *>(aPrev + r * LD + i) =
                            make_float4(d[e][v * 4 + 0], d[e][v * 4 + 1], d[e][v * 4 + 2], d[e][v * 4 + 3]);
                }
            __syncthreads();
        }
        // ---- layer 1: sAct[0] holds dz_0[r][i]
        if (tid < H) {
            float s1 = 0.f, s0 = 0.f;
            for (int r = 0; r < TM; ++r) {
                const float v = sAct[r * LD + tid];
                s0 += v;
                s1 = fmaf(v, sX[r], s1);
            }
            pw1 += s1;
            pb1 += s0;
        }
        if (a.du && row0 + tid < a.R) {  // du[r,g] = sum_i dz_0[r][i] * w1[i]   (row tid; rotated start: no bank conflicts)
            float s = 0.f;
            for (int k = 0; k < H; ++k) {
                const int i = (k + tid) & (H - 1);
                s = fmaf(sAct[tid * LD + i], sW1[i], s);
            }
            a.du[(row0 + tid) * a.G + g] = s;
        }
    }
    __syncthreads();
    // ---- write this CTA's partial gradients
    const size_t off = (size_t)blockIdx.x * gp.chunk_stride;
    if (tid < H) {
        if (gp.w1) gp.w1[off + (size_t)g * H + tid] = pw1;
        if (gp.b1) gp.b1[off + (size_t)g * H + tid] = pb1;
#pragma unroll
        for (int l = 0; l < NH; ++l)
            if (gp.bh) gp.bh[off + ((size_t)l * a.G + g) * H + tid] = pbh[l];
    }
    if (tid < a.C && gp.bo) gp.bo[off + (size_t)g * a.C + tid] = pbo;
    if (gp.wo)
        for (int i = tid; i < a.C * H; i += NT) gp.wo[off + (size_t)g * a.C * H + i] = sDWo[(i / H) * LD + (i % H)];
    if (gp.wh && ty2 * 8 < H && tx2 * 4 < H) {
#pragma unroll
        for (int l = 0; l < NH; ++l)
#pragma unroll
            for (int e = 0; e < 8; ++e)
                *reinterpret_cast<float4 *>(gp.wh + off + (((size_t)l * a.G + g) * H + ty2 * 8 + e) * H + tx2 * 4) =
                    make_float4(accW[l][e][0], accW[l][e][1], accW[l][e][2], accW[l][e][3]);
    }
}

// ---- n_layers == 1: f_g(u) = wo[g,:,0]*u + bo[g] --------------------------------------------------------------
__global__ void linear1_fwd_kernel(MlpKArgs a, float *__restrict__ S)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.R * a.C) return;
    const int64_t r = i / a.C;
    const int c = (int)(i % a.C);
    float s = 0.f;
    for (int g = 0; g < a.G; ++g) s += fmaf(a.u[r * a.ldu + g], a.wo[(size_t)g * a.C + c], a.bo ? a.bo[(size_t)g * a.C + c] : 0.f);
    S[i] = s;
}

// one block per (g); threads reduce over rows
__global__ void linear1_bwd_kernel(MlpKArgs a, const float *__restrict__ dS, float *__restrict__ dwo, float *__restrict__ dbo)
{
    __shared__ float red[2][256];
    const int g = blockIdx.x;
    for (int c = 0; c < a.C; ++c) {
        float sw = 0.f, sb = 0.f;
        for (int64_t r = threadIdx.x; r < a.R; r += blockDim.x) {
            const float gv = dS[r * a.C + c];
            sw = fmaf(gv, a.u[r * a.ldu + g], sw);
            sb += gv;
        }
        red[0][threadIdx.x] = sw;
        red[1][threadIdx.x] = sb;
        __syncthreads();
        for (int s = blockDim.x / 2; s > 0; s >>= 1) {
            if ((int)threadIdx.x < s) {
                red[0][threadIdx.x] += red[0][threadIdx.x + s];
                red[1][threadIdx.x] += red[1][threadIdx.x + s];
            }
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            if (dwo) dwo[(size_t)g * a.C + c] = red[0][0];
            if (dbo) dbo[(size_t)g * a.C + c] = red[1][0];
        }
        __syncthreads();
    }
}

// du[r,g] = sum_c dS[r,c] * wo[g,c]
__global__ void linear1_du_kernel(MlpKArgs a, const float *__restrict__ dS)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.R * a.G) return;
    const int64_t r = i / a.G;
    const int g = (int)(i % a.G);
    float s = 0.f;
    for (int c = 0; c < a.C; ++c) s = fmaf(dS[r * a.C + c], a.wo[(size_t)g * a.C + c], s);
    a.du[i] = s;
}

// ---- host side ------------------------------------------------------------------------------------------------
inline size_t pad4(size_t n) { return (n + 3) / 4 * 4; }

// floats of one partial-gradient chunk; every segment starts 16-byte aligned (the kernel stores float4s)
// ---- entries mode, SMALL groups (bag-of-words columns: a few dozen distinct values per feature): one CTA per feature ----------
// The tcgen05 backward stages 64 KB of split weights, allocates tensor memory and drains its pipeline once per (feature, tile):
// with ~35 rows per feature that set-up is the whole cost (Cora shape: 1 434 CTAs, one per SM at a time, 15 us each). Here a
// feature is a 256-thread CTA with 46 KB of shared memory (4-5 CTAs per SM overlap each other's latencies), plain fp32 FMAs:
// 32-row tiles, W2 in shared memory with an odd row stride (65: conflict free along rows and columns), dW2 as a 4x4 register
// block per thread, every gradient of the feature written straight to its place (no partial chunks, no reduction kernel).
constexpr int SG_RT = 32, SG_LD = 65, SG_THREADS = 256, SG_H = 64, SG_C = 8;
constexpr int SG_AVG_MAX = 96;                           // used when a feature has at most this many entries on average
constexpr int SG_GROUP_MAX = 32 * SG_AVG_MAX;            // ... and no single feature more than this (one CTA walks a feature's tiles serially)

__global__ void __launch_bounds__(SG_THREADS, 3)
mlp_entries_bwd_small_kernel(MlpKArgs a, const float *__restrict__ dY, MlpGradPtrs gp)
{
    __shared__ float sW[SG_H * SG_LD], sA0[SG_RT * SG_LD], sA1[SG_RT * SG_LD], sDz[SG_RT * SG_LD];
    __shared__ float sG[SG_RT * SG_C], sX[SG_RT], sW1[SG_H], sB1[SG_H], sB2[SG_H], sWo[SG_C * SG_H];
    const int tid = threadIdx.x, t16 = tid & 15, r2 = tid >> 4, g = blockIdx.x, C = a.C;
    const int64_t ebase = a.grp_ptr[g], nrow = a.grp_ptr[g + 1] - ebase;
    {
        const float *W = a.wh + (size_t)g * SG_H * SG_H;
        for (int idx = tid; idx < SG_H * SG_H; idx += SG_THREADS) sW[(idx >> 6) * SG_LD + (idx & 63)] = __ldg(W + idx);
        if (tid < SG_H) {
            sW1[tid] = __ldg(a.w1 + (size_t)g * SG_H + tid);
            sB1[tid] = a.b1 ? __ldg(a.b1 + (size_t)g * SG_H + tid) : 0.f;
            sB2[tid] = a.bh ? __ldg(a.bh + (size_t)g * SG_H + tid) : 0.f;
        }
        for (int idx = tid; idx < SG_C * SG_H; idx += SG_THREADS) {
            const int c = idx >> 6;
            sWo[idx] = c < C ? __ldg(a.wo + ((size_t)g * C + c) * SG_H + (idx & 63)) : 0.f;
        }
    }
    float accW[4][4];                                    // dW2[r2*4 + q][t16 + 16 p]
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int pp = 0; pp < 4; ++pp) accW[q][pp] = 0.f;
    float wo0 = 0.f, wo1 = 0.f;                          // dWo[c = warp][lane], [lane + 32]
    float pb2 = 0.f, pw1 = 0.f, pb1 = 0.f, pbo = 0.f;    // column sums owned by tid < 64 (bo: tid 64..71)
    const int rA = 2 * r2, rB = rA + 1;
    for (int64_t row0 = 0; row0 < nrow; row0 += SG_RT) {
        __syncthreads();                                 // previous tile consumed (first pass: the weights are staged)
        if (tid < SG_RT) sX[tid] = row0 + tid < nrow ? __ldg(a.u + ebase + row0 + tid) : 0.f;
        {
            const int r = tid >> 3, c = tid & 7;
            sG[tid] = (row0 + r < nrow && c < C) ? __ldg(dY + (ebase + row0 + r) * C + c) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int e = 0; e < SG_RT * SG_H / SG_THREADS; ++e) {
            const int idx = tid + SG_THREADS * e, r = idx >> 6, i = idx & 63;
            sA0[r * SG_LD + i] = relu(fmaf(sX[r], sW1[i], sB1[i]));
        }
        __syncthreads();
        {   // z2 = a0 W2^T + b2 for rows rA, rB and units t16 + 16 q; then a1, dh = g Wo, dz2
            float acc[2][4];
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[0][q] = acc[1][q] = sB2[t16 + 16 * q];
#pragma unroll 8
            for (int i = 0; i < SG_H; ++i) {
                const float xa = sA0[rA * SG_LD + i], xb = sA0[rB * SG_LD + i];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float w = sW[(t16 + 16 * q) * SG_LD + i];
                    acc[0][q] = fmaf(xa, w, acc[0][q]);
                    acc[1][q] = fmaf(xb, w, acc[1][q]);
                }
            }
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int r = rA + h;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int j = t16 + 16 * q;
                    float dh = 0.f;
#pragma unroll
                    for (int c = 0; c < SG_C; ++c) dh = fmaf(sG[r * SG_C + c], sWo[c * SG_H + j], dh);
                    const float z = acc[h][q];
                    sA1[r * SG_LD + j] = relu(z);
                    sDz[r * SG_LD + j] = z > 0.f ? dh : 0.f;
                }
            }
        }
        __syncthreads();
        // dW2[j][i] += sum_r dz2[r][j] a0[r][i]
#pragma unroll 4
        for (int r = 0; r < SG_RT; ++r) {
            float dz[4], av[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) { dz[q] = sDz[r * SG_LD + r2 * 4 + q]; av[q] = sA0[r * SG_LD + t16 + 16 * q]; }
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
                for (int pp = 0; pp < 4; ++pp) accW[q][pp] = fmaf(dz[q], av[pp], accW[q][pp]);
        }
        {   // dWo[c][j] += sum_r g[r][c] a1[r][j]: a warp per channel
            const int c = tid >> 5, jj = tid & 31;
#pragma unroll 8
            for (int r = 0; r < SG_RT; ++r) {
                const float gv = sG[r * SG_C + c];
                wo0 = fmaf(gv, sA1[r * SG_LD + jj], wo0);
                wo1 = fmaf(gv, sA1[r * SG_LD + jj + 32], wo1);
            }
        }
        if (tid < SG_H) {
#pragma unroll 8
            for (int r = 0; r < SG_RT; ++r) pb2 += sDz[r * SG_LD + tid];
        } else if (tid < SG_H + SG_C) {
#pragma unroll 8
            for (int r = 0; r < SG_RT; ++r) pbo += sG[r * SG_C + tid - SG_H];
        }
        float dz1[2][4];
        {   // da0 = dz2 W2 for rows rA, rB and units t16 + 16 q; dz1 = da0 * 1[a0 > 0]
            float acc[2][4];
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[0][q] = acc[1][q] = 0.f;
#pragma unroll 8
            for (int j = 0; j < SG_H; ++j) {
                const float da = sDz[rA * SG_LD + j], db = sDz[rB * SG_LD + j];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float w = sW[j * SG_LD + t16 + 16 * q];
                    acc[0][q] = fmaf(da, w, acc[0][q]);
                    acc[1][q] = fmaf(db, w, acc[1][q]);
                }
            }
#pragma unroll
            for (int h = 0; h < 2; ++h)
#pragma unroll
                for (int q = 0; q < 4; ++q) dz1[h][q] = sA0[(rA + h) * SG_LD + t16 + 16 * q] > 0.f ? acc[h][q] : 0.f;
        }
        __syncthreads();                                 // a1 (dWo) and dz2 are consumed: a1's buffer takes dz1
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int q = 0; q < 4; ++q) sA1[(rA + h) * SG_LD + t16 + 16 * q] = dz1[h][q];
        __syncthreads();
        if (tid < SG_H) {
#pragma unroll 8
            for (int r = 0; r < SG_RT; ++r) {
                const float d = sA1[r * SG_LD + tid];
                pw1 = fmaf(d, sX[r], pw1);
                pb1 += d;
            }
        }
    }
    if (gp.wh) {
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
            for (int pp = 0; pp < 4; ++pp) gp.wh[((size_t)g * SG_H + r2 * 4 + q) * SG_H + t16 + 16 * pp] = accW[q][pp];
    }
    {
        const int c = tid >> 5, jj = tid & 31;
        if (gp.wo && c < C) {
            gp.wo[((size_t)g * C + c) * SG_H + jj] = wo0;
            gp.wo[((size_t)g * C + c) * SG_H + jj + 32] = wo1;
        }
    }
    if (tid < SG_H) {
        if (gp.bh) gp.bh[(size_t)g * SG_H + tid] = pb2;
        if (gp.w1) gp.w1[(size_t)g * SG_H + tid] = pw1;
        if (gp.b1) gp.b1[(size_t)g * SG_H + tid] = pb1;
    } else if (tid < SG_H + C) {
        if (gp.bo) gp.bo[(size_t)g * C + tid - SG_H] = pbo;
    }
}

size_t grad_floats(const gnan_mlp_params *p)
{
    const size_t G = p->G, H = p->H, C = p->C, nh = p->n_layers - 2;
    return 2 * pad4(G * H) + pad4(nh * G * H * H) + pad4(nh * G * H) + pad4(G * C * H) + pad4(G * C);
}

struct FwdPlan { int KC; int nchunk; int64_t ntile; size_t smem; };

FwdPlan plan_fwd(int64_t R, const gnan_mlp_params *p)
{
    FwdPlan pl;
    pl.ntile = ceil_div64(R, TM);
    const int target = 2 * 3 * gnan_sm_count();  // ~2 waves at 3 CTAs/SM
    int nchunk = (int)ceil_div64(target, pl.ntile);
    if (nchunk < 1) nchunk = 1;
    int KC = (int)ceil_div64(p->G, nchunk);
    if (KC < 8) KC = p->G < 8 ? p->G : 8;   // keep x-tile loads sector-efficient
    if (KC > 32) KC = 32;
    pl.KC = KC;
    pl.nchunk = (int)ceil_div64(p->G, KC);
    const int H = p->H, LD = H + 4, CP = (p->C + 7) / 8 * 8;
    pl.smem = sizeof(float) * ((size_t)TM * LD + (size_t)H * LD + (size_t)CP * LD + (size_t)TM * CP + (size_t)KC * TM + 3 * H + CP);
    return pl;
}

struct BwdPlan { int nchunk; int64_t ntile; size_t smem; };

BwdPlan plan_bwd(int64_t R, const gnan_mlp_params *p)
{
    BwdPlan pl;
    pl.ntile = ceil_div64(R, TM);
    const int nh = p->n_layers - 2;
    const int per_sm = (p->H <= 64 && nh <= 1) ? 2 : 1;
    const int target = 2 * per_sm * gnan_sm_count();
    int nchunk = (int)ceil_div64(target, p->G);
    nchunk = (int)std::min<int64_t>(nchunk, std::max<int64_t>(1, pl.ntile / 4));   // >= 4 tiles per CTA: short partial reduction
    if (nchunk < 1) nchunk = 1;
    pl.nchunk = nchunk;
    const int H = p->H, LD = H + 4, CP = (p->C + 7) / 8 * 8, CG = CP + 4;
    const int nha = nh > 0 ? nh : 1;
    pl.smem = sizeof(float) * ((size_t)(nh + 1) * TM * LD + (size_t)H * LD + 2 * (size_t)CP * LD + (size_t)TM * CG + TM + 2 * H + (size_t)nha * H);
    return pl;
}

int check_params(const gnan_mlp_params *p, int64_t R, int64_t ldu)
{
    GNAN_REQUIRE(p != nullptr, "mlp: params is NULL");
    GNAN_REQUIRE(p->G >= 1 && p->C >= 1 && p->n_layers >= 1, "mlp: need G,C,n_layers >= 1 (got %d,%d,%d)", p->G, p->C, p->n_layers);
    GNAN_REQUIRE(R >= 0 && ldu >= p->G, "mlp: need R >= 0 and ldu >= G (R=%lld ldu=%lld G=%d)", (long long)R, (long long)ldu, p->G);
    GNAN_REQUIRE(p->wo != nullptr, "mlp: wo is NULL");
    if (p->n_layers >= 2) {
        GNAN_REQUIRE(p->w1 != nullptr, "mlp: w1 is NULL");
        GNAN_REQUIRE(p->n_layers == 2 || p->wh != nullptr, "mlp: wh is NULL with n_layers=%d", p->n_layers);
        if (!(p->H == 8 || p->H == 16 || p->H == 32 || p->H == 64)) {
            gnan_set_error("mlp: hidden width %d unsupported (8,16,32,64)", p->H);
            return GNAN_ERR_UNSUPPORTED;
        }
        if (p->n_layers > 5) {
            gnan_set_error("mlp: n_layers %d unsupported (<= 5)", p->n_layers);
            return GNAN_ERR_UNSUPPORTED;
        }
        if (p->C > 64) {
            gnan_set_error("mlp: out_channels %d unsupported (<= 64)", p->C);
            return GNAN_ERR_UNSUPPORTED;
        }
    }
    return GNAN_OK;
}

MlpKArgs make_args(const float *u, int64_t R, int64_t ldu, const gnan_mlp_params *p, float dropout_p, uint64_t seed)
{
    MlpKArgs a;
    a.u = u; a.R = R; a.ldu = ldu; a.G = p->G; a.C = p->C; a.nh = p->n_layers - 2;
    a.w1 = p->w1; a.b1 = p->b1; a.wh = p->wh; a.bh = p->bh; a.wo = p->wo; a.bo = p->bo;
    a.drop_thresh = dropout_p > 0.f ? gnan_dropout_thresh(dropout_p) : 0u;
    a.drop_scale = dropout_p > 0.f ? 1.f / (1.f - dropout_p) : 1.f;
    a.seed = seed;
    a.seed_dev = nullptr;
    a.du = nullptr;
    a.grp_ptr = nullptr;
    a.items = nullptr;
    return a;
}

template <int H>
int launch_fwd(const MlpKArgs &a, const FwdPlan &pl, float *Spart, cudaStream_t st)
{
    GNAN_CUDA(cudaFuncSetAttribute(mlp_fwd_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
    dim3 grid((unsigned)pl.ntile, (unsigned)pl.nchunk);
    mlp_fwd_kernel<H><<<grid, NT, pl.smem, st>>>(a, pl.KC, Spart);
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}

template <int H, int NH>
int launch_bwd(const MlpKArgs &a, const BwdPlan &pl, const float *dS, const MlpGradPtrs &gp, cudaStream_t st)
{
    GNAN_CUDA(cudaFuncSetAttribute(mlp_bwd_kernel<H, NH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
    dim3 grid((unsigned)pl.nchunk, (unsigned)a.G);
    mlp_bwd_kernel<H, NH><<<grid, NT, pl.smem, st>>>(a, dS, gp, pl.ntile);
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}

template <int H>
int launch_bwd_h(const MlpKArgs &a, const BwdPlan &pl, const float *dS, const MlpGradPtrs &gp, cudaStream_t st)
{
    switch (a.nh) {
        case 0: return launch_bwd<H, 0>(a, pl, dS, gp, st);
        case 1: return launch_bwd<H, 1>(a, pl, dS, gp, st);
        case 2: return launch_bwd<H, 2>(a, pl, dS, gp, st);
        case 3: return launch_bwd<H, 3>(a, pl, dS, gp, st);
    }
    gnan_set_error("mlp_bwd: n_hidden %d unsupported", a.nh);
    return GNAN_ERR_UNSUPPORTED;
}

}  // namespace

// tcgen05 path (mlp_tc.cu)
int gnan_mlp_tc_supported(const gnan_mlp_params *p, int precision);
int gnan_mlp_tc_bwd_supported(const gnan_mlp_params *p, int precision);
size_t gnan_mlp_tc_workspace_bytes(int64_t R, const gnan_mlp_params *p, int backward, int precision);
int gnan_mlp_tc_fwd(const float *u, int64_t R, int64_t ldu, const gnan_mlp_params *p, float dropout_p, uint64_t seed,
                    int precision, float *S, void *ws, size_t ws_bytes, cudaStream_t st, const uint64_t *seed_dev);
int gnan_mlp_tc_entries_fwd_supported(const gnan_mlp_params *p, int precision);
int gnan_mlp_tc_entries_fwd(const float *val, const int64_t *grp_ptr, int64_t E, const int32_t *items, int64_t n_items,
                            const gnan_mlp_params *p, int precision, float *Y, cudaStream_t st);
int gnan_mlp_tc_bwd_ex(const float *u, int64_t R, int64_t ldu, const gnan_mlp_params *p, float dropout_p, uint64_t seed,
                       int precision, const float *dS, const gnan_mlp_grads *grads, void *ws, size_t ws_bytes, cudaStream_t st,
                       const int64_t *grp_ptr, const uint64_t *seed_dev, const float *dh_ext, float *a1_ext);

extern "C" size_t gnan_mlp_workspace_bytes(int64_t R, const gnan_mlp_params *p, int backward, int precision)
{
    if (!p || p->n_layers < 2 || R <= 0) return 0;
    if (precision != GNAN_PREC_FP32 && (backward ? gnan_mlp_tc_bwd_supported(p, precision) : gnan_mlp_tc_supported(p, precision)))
        return gnan_mlp_tc_workspace_bytes(R, p, backward, precision);
    if (!backward) {
        const FwdPlan pl = plan_fwd(R, p);
        return pl.nchunk > 1 ? sizeof(float) * (size_t)pl.nchunk * R * p->C : 0;
    }
    const BwdPlan pl = plan_bwd(R, p);
    return pl.nchunk > 1 ? sizeof(float) * (size_t)pl.nchunk * grad_floats(p) : 0;
}

extern "C" int gnan_mlp_fwd(const float *u, int64_t R, int64_t ldu, const gnan_mlp_params *p, float dropout_p,
                            uint64_t seed, const uint64_t *seed_dev, int precision, float *S, void *workspace,
                            size_t workspace_bytes, gnan_stream_t stream)
{
    int rc = check_params(p, R, ldu);
    if (rc) return rc;
    GNAN_REQUIRE(S != nullptr && (u != nullptr || R == 0), "mlp_fwd: NULL u or S");
    GNAN_REQUIRE(dropout_p >= 0.f && dropout_p < 1.f, "mlp_fwd: dropout_p %f out of [0,1)", dropout_p);
    cudaStream_t st = (cudaStream_t)stream;
    if (R == 0) return GNAN_OK;
    MlpKArgs a = make_args(u, R, ldu, p, dropout_p, seed);
    a.seed_dev = dropout_p > 0.f ? seed_dev : nullptr;
    if (p->n_layers == 1) {
        const int64_t n = R * p->C;
        linear1_fwd_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, st>>>(a, S);
        GNAN_LAUNCH_OK();
        return GNAN_OK;
    }
    // shapes the tensor-core path does not cover run the (more precise) fp32 kernel
    if (precision != GNAN_PREC_FP32 && gnan_mlp_tc_supported(p, precision))
        return gnan_mlp_tc_fwd(u, R, ldu, p, dropout_p, seed, precision, S, workspace, workspace_bytes, st, a.seed_dev);
    const FwdPlan pl = plan_fwd(R, p);
    float *Spart = S;
    if (pl.nchunk > 1) {
        const size_t need = sizeof(float) * (size_t)pl.nchunk * R * p->C;
        if (workspace == nullptr || workspace_bytes < need) {
            gnan_set_error("mlp_fwd: workspace %zu < %zu bytes", workspace_bytes, need);
            return GNAN_ERR_WORKSPACE;
        }
        Spart = (float *)workspace;
    }
    switch (p->H) {
        case 8: rc = launch_fwd<8>(a, pl, Spart, st); break;
        case 16: rc = launch_fwd<16>(a, pl, Spart, st); break;
        case 32: rc = launch_fwd<32>(a, pl, Spart, st); break;
        case 64: rc = launch_fwd<64>(a, pl, Spart, st); break;
    }
    if (rc) return rc;
    if (pl.nchunk > 1) {
        const size_t n = (size_t)R * p->C;
        rc = gnan_reduce_chunks(Spart, pl.nchunk, n, n, S, st);
        if (rc) return rc;
    }
    return GNAN_OK;
}

static int mlp_bwd_impl(const float *u, int64_t R, int64_t ldu, const gnan_mlp_params *p, float dropout_p,
                        uint64_t seed, const uint64_t *seed_dev, int precision, const float *dS, const gnan_mlp_grads *grads,
                        void *workspace, size_t workspace_bytes, gnan_stream_t stream, const float *dh_ext, float *a1_ext);

extern "C" int gnan_mlp_bwd(const float *u, int64_t R, int64_t ldu, const gnan_mlp_params *p, float dropout_p,
                            uint64_t seed, const uint64_t *seed_dev, int precision, const float *dS, const gnan_mlp_grads *grads,
                            void *workspace, size_t workspace_bytes, gnan_stream_t stream)
{
    return mlp_bwd_impl(u, R, ldu, p, dropout_p, seed, seed_dev, precision, dS, grads, workspace, workspace_bytes, stream, nullptr, nullptr);
}

// 1 when gnan_mlp_bwd_ext covers the shape: the tcgen05 backward (H = 64, 3 layers) with more than 8 output channels
extern "C" int gnan_mlp_bwd_ext_supported(const gnan_mlp_params *p, int precision)
{
    return p && precision != GNAN_PREC_FP32 && gnan_mlp_tc_bwd_supported(p, precision) && p->C > 8;
}

extern "C" int gnan_mlp_bwd_ext(const float *u, int64_t R, int64_t ldu, const gnan_mlp_params *p, float dropout_p, uint64_t seed,
                                const uint64_t *seed_dev, int precision, const float *dS, const float *dh, float *a1,
                                const gnan_mlp_grads *grads, void *workspace, size_t workspace_bytes, gnan_stream_t stream)
{
    GNAN_REQUIRE(p && gnan_mlp_bwd_ext_supported(p, precision), "mlp_bwd_ext: needs the tensor-core backward (H = 64, 3 layers, precision != fp32) and C > 8");
    GNAN_REQUIRE(grads && grads->du == nullptr && grads->wo == nullptr, "mlp_bwd_ext: du is not available and dWo is the caller's GEMM (pass NULL)");
    GNAN_REQUIRE(R == 0 || (dh && a1), "mlp_bwd_ext: NULL dh / a1");
    return mlp_bwd_impl(u, R, ldu, p, dropout_p, seed, seed_dev, precision, dS, grads, workspace, workspace_bytes, stream, dh, a1);
}

static int mlp_bwd_impl(const float *u, int64_t R, int64_t ldu, const gnan_mlp_params *p, float dropout_p,
                        uint64_t seed, const uint64_t *seed_dev, int precision, const float *dS, const gnan_mlp_grads *grads,
                        void *workspace, size_t workspace_bytes, gnan_stream_t stream, const float *dh_ext, float *a1_ext)
{
    int rc = check_params(p, R, ldu);
    if (rc) return rc;
    GNAN_REQUIRE(grads != nullptr && (R == 0 || (u != nullptr && dS != nullptr)), "mlp_bwd: NULL u, dS or grads");
    GNAN_REQUIRE(dropout_p >= 0.f && dropout_p < 1.f, "mlp_bwd: dropout_p %f out of [0,1)", dropout_p);
    cudaStream_t st = (cudaStream_t)stream;
    MlpKArgs a = make_args(u, R, ldu, p, dropout_p, seed);
    a.seed_dev = dropout_p > 0.f ? seed_dev : nullptr;
    a.du = grads->du;
    const size_t G = p->G, H = p->H, C = p->C;
    if (p->n_layers == 1) {
        linear1_bwd_kernel<<<p->G, 256, 0, st>>>(a, dS, grads->wo, grads->bo);
        GNAN_LAUNCH_OK();
        if (a.du && R > 0) {
            linear1_du_kernel<<<(unsigned)ceil_div64(R * p->G, 256), 256, 0, st>>>(a, dS);
            GNAN_LAUNCH_OK();
        }
        return GNAN_OK;
    }
    const size_t nh = p->n_layers - 2;
    if (R == 0) {
        if (grads->w1) GNAN_CUDA(cudaMemsetAsync(grads->w1, 0, sizeof(float) * G * H, st));
        if (grads->b1) GNAN_CUDA(cudaMemsetAsync(grads->b1, 0, sizeof(float) * G * H, st));
        if (grads->wh && nh) GNAN_CUDA(cudaMemsetAsync(grads->wh, 0, sizeof(float) * nh * G * H * H, st));
        if (grads->bh && nh) GNAN_CUDA(cudaMemsetAsync(grads->bh, 0, sizeof(float) * nh * G * H, st));
        if (grads->wo) GNAN_CUDA(cudaMemsetAsync(grads->wo, 0, sizeof(float) * G * C * H, st));
        if (grads->bo) GNAN_CUDA(cudaMemsetAsync(grads->bo, 0, sizeof(float) * G * C, st));
        return GNAN_OK;
    }
    if (precision != GNAN_PREC_FP32 && !grads->du && gnan_mlp_tc_bwd_supported(p, precision))   // input gradients: fp32 kernel only
        return gnan_mlp_tc_bwd_ex(u, R, ldu, p, dropout_p, seed, precision, dS, grads, workspace, workspace_bytes, st, nullptr, a.seed_dev, dh_ext, a1_ext);
    const BwdPlan pl = plan_bwd(R, p);
    MlpGradPtrs gp;
    const size_t ntot = grad_floats(p);
    if (pl.nchunk > 1) {
        const size_t need = sizeof(float) * (size_t)pl.nchunk * ntot;
        if (workspace == nullptr || workspace_bytes < need) {
            gnan_set_error("mlp_bwd: workspace %zu < %zu bytes", workspace_bytes, need);
            return GNAN_ERR_WORKSPACE;
        }
        float *w = (float *)workspace;
        gp.w1 = w; w += pad4(G * H);
        gp.b1 = w; w += pad4(G * H);
        gp.wh = w; w += pad4(nh * G * H * H);
        gp.bh = w; w += pad4(nh * G * H);
        gp.wo = w; w += pad4(G * C * H);
        gp.bo = w;
        gp.chunk_stride = ntot;
    } else {
        gp.w1 = grads->w1; gp.b1 = grads->b1; gp.wh = grads->wh; gp.bh = grads->bh; gp.wo = grads->wo; gp.bo = grads->bo;
        gp.chunk_stride = 0;
    }
    switch (p->H) {
        case 8: rc = launch_bwd_h<8>(a, pl, dS, gp, st); break;
        case 16: rc = launch_bwd_h<16>(a, pl, dS, gp, st); break;
        case 32: rc = launch_bwd_h<32>(a, pl, dS, gp, st); break;
        case 64: rc = launch_bwd_h<64>(a, pl, dS, gp, st); break;
    }
    if (rc) return rc;
    if (pl.nchunk > 1) {
        GnanReduceSegs sg{};                                    // all six gradient arrays in one launch
        sg.add(gp.w1, grads->w1, G * H); sg.add(gp.b1, grads->b1, G * H); sg.add(gp.wh, grads->wh, nh * G * H * H);
        sg.add(gp.bh, grads->bh, nh * G * H); sg.add(gp.wo, grads->wo, G * C * H); sg.add(gp.bo, grads->bo, G * C);
        rc = gnan_reduce_chunks_multi(sg, pl.nchunk, ntot, st);
        if (rc) return rc;
    }
    return GNAN_OK;
}


// ---- entries mode: shape functions on a compressed feature matrix ---------------------------------------------------
// A feature column that repeats one value (zeros of a bag-of-words matrix, the off entries of a one-hot encoding, the
// constant column) needs ONE evaluation for that value when dropout is off; only the other entries need their own. The
// caller lists the distinct work as `val[E]` grouped by feature (`grp_ptr[G+1]`) and gets Y[e,:] = f_g(val[e]) back.
namespace {
int check_entries(const gnan_mlp_params *p, const float *val, const int64_t *grp_ptr, int64_t E, const char *who)
{
    int rc = check_params(p, E, p ? p->G : 1);
    if (rc) return rc;
    GNAN_REQUIRE(p->n_layers >= 2, "%s: n_layers == 1 has no entries mode (a Linear(1,C) is cheaper evaluated densely)", who);
    GNAN_REQUIRE(E >= 0 && (E == 0 || val != nullptr) && grp_ptr != nullptr, "%s: NULL val or grp_ptr", who);
    return GNAN_OK;
}
}  // namespace

extern "C" size_t gnan_mlp_entries_workspace_bytes(int64_t max_group_entries, const gnan_mlp_params *p, int backward, int precision)
{
    if (!p || p->n_layers < 2 || max_group_entries <= 0 || !backward) return 0;
    if (precision != GNAN_PREC_FP32 && gnan_mlp_tc_bwd_supported(p, precision))
        return gnan_mlp_tc_workspace_bytes(max_group_entries, p, 1, precision);
    const BwdPlan pl = plan_bwd(max_group_entries, p);
    return pl.nchunk > 1 ? sizeof(float) * (size_t)pl.nchunk * grad_floats(p) : 0;
}

extern "C" int gnan_mlp_entries_fwd_ex(const float *val, const int64_t *grp_ptr, int64_t E, const int32_t *items, int64_t n_items,
                                       const gnan_mlp_params *p, int precision, float *Y, gnan_stream_t stream)
{
    int rc = check_entries(p, val, grp_ptr, E, "mlp_entries_fwd");
    if (rc) return rc;
    GNAN_REQUIRE(n_items >= 0 && (n_items == 0 || (items != nullptr && Y != nullptr)), "mlp_entries_fwd: NULL items or Y");
    if (n_items == 0) return GNAN_OK;
    if (precision != GNAN_PREC_FP32 && gnan_mlp_tc_entries_fwd_supported(p, precision))      // tcgen05 kernel
        return gnan_mlp_tc_entries_fwd(val, grp_ptr, E, items, n_items, p, precision, Y, (cudaStream_t)stream);
    MlpKArgs a = make_args(val, E, 1, p, 0.f, 0);
    a.grp_ptr = grp_ptr;
    a.items = items;
    FwdPlan pl;
    pl.KC = 1; pl.nchunk = 1; pl.ntile = n_items;
    const int H = p->H, LD = H + 4, CP = (p->C + 7) / 8 * 8;
    pl.smem = sizeof(float) * ((size_t)TM * LD + (size_t)H * LD + (size_t)CP * LD + (size_t)TM * CP + (size_t)TM + 3 * H + CP);
    cudaStream_t st = (cudaStream_t)stream;
    switch (p->H) {
        case 8: return launch_fwd<8>(a, pl, Y, st);
        case 16: return launch_fwd<16>(a, pl, Y, st);
        case 32: return launch_fwd<32>(a, pl, Y, st);
        case 64: return launch_fwd<64>(a, pl, Y, st);
    }
    return GNAN_ERR_UNSUPPORTED;
}

extern "C" int gnan_mlp_entries_bwd(const float *val, const int64_t *grp_ptr, int64_t E, int64_t max_group_entries,
                                    const gnan_mlp_params *p, int precision, const float *dY, const gnan_mlp_grads *grads,
                                    void *workspace, size_t workspace_bytes, gnan_stream_t stream)
{
    int rc = check_entries(p, val, grp_ptr, E, "mlp_entries_bwd");
    if (rc) return rc;
    GNAN_REQUIRE(grads != nullptr && (E == 0 || dY != nullptr), "mlp_entries_bwd: NULL dY or grads");
    GNAN_REQUIRE(grads->du == nullptr, "mlp_entries_bwd: input gradients are not available in entries mode");
    GNAN_REQUIRE(max_group_entries >= 0 && max_group_entries <= E, "mlp_entries_bwd: bad max_group_entries");
    cudaStream_t st = (cudaStream_t)stream;
    if (E > 0 && p->H == SG_H && p->n_layers == 3 && p->C <= SG_C && E <= (int64_t)SG_AVG_MAX * p->G && max_group_entries <= SG_GROUP_MAX) {
        // few rows per feature (bag-of-words columns): a CTA per feature on the CUDA cores, fp32 (both precision modes)
        MlpKArgs a = make_args(val, E, 1, p, 0.f, 0);
        a.grp_ptr = grp_ptr;
        MlpGradPtrs gp;
        gp.w1 = grads->w1; gp.b1 = grads->b1; gp.wh = grads->wh; gp.bh = grads->bh; gp.wo = grads->wo; gp.bo = grads->bo;
        gp.chunk_stride = 0;
        mlp_entries_bwd_small_kernel<<<(unsigned)p->G, SG_THREADS, 0, st>>>(a, dY, gp);
        GNAN_LAUNCH_OK();
        return GNAN_OK;
    }
    if (E > 0 && precision != GNAN_PREC_FP32 && gnan_mlp_tc_bwd_supported(p, precision))      // tcgen05 kernel, per-group row space
        return gnan_mlp_tc_bwd_ex(val, std::max<int64_t>(max_group_entries, 1), 1, p, 0.f, 0, precision, dY, grads, workspace,
                                  workspace_bytes, st, grp_ptr, nullptr, nullptr, nullptr);
    MlpKArgs a = make_args(val, E, 1, p, 0.f, 0);
    a.grp_ptr = grp_ptr;
    const size_t G = p->G, H = p->H, C = p->C, nh = p->n_layers - 2;
    const BwdPlan pl = plan_bwd(std::max<int64_t>(max_group_entries, 1), p);   // groups without entries write zero gradients
    MlpGradPtrs gp;
    const size_t ntot = grad_floats(p);
    if (pl.nchunk > 1) {
        const size_t need = sizeof(float) * (size_t)pl.nchunk * ntot;
        if (workspace == nullptr || workspace_bytes < need) {
            gnan_set_error("mlp_entries_bwd: workspace %zu < %zu bytes", workspace_bytes, need);
            return GNAN_ERR_WORKSPACE;
        }
        float *w = (float *)workspace;
        gp.w1 = w; w += pad4(G * H);
        gp.b1 = w; w += pad4(G * H);
        gp.wh = w; w += pad4(nh * G * H * H);
        gp.bh = w; w += pad4(nh * G * H);
        gp.wo = w; w += pad4(G * C * H);
        gp.bo = w;
        gp.chunk_stride = ntot;
    } else {
        gp.w1 = grads->w1; gp.b1 = grads->b1; gp.wh = grads->wh; gp.bh = grads->bh; gp.wo = grads->wo; gp.bo = grads->bo;
        gp.chunk_stride = 0;
    }
    switch (p->H) {
        case 8: rc = launch_bwd_h<8>(a, pl, dY, gp, st); break;
        case 16: rc = launch_bwd_h<16>(a, pl, dY, gp, st); break;
        case 32: rc = launch_bwd_h<32>(a, pl, dY, gp, st); break;
        case 64: rc = launch_bwd_h<64>(a, pl, dY, gp, st); break;
    }
    if (rc) return rc;
    if (pl.nchunk > 1) {
        GnanReduceSegs sg{};
        sg.add(gp.w1, grads->w1, G * H); sg.add(gp.b1, grads->b1, G * H); sg.add(gp.wh, grads->wh, nh * G * H * H);
        sg.add(gp.bh, grads->bh, nh * G * H); sg.add(gp.wo, grads->wo, G * C * H); sg.add(gp.bo, grads->bo, G * C);
        rc = gnan_reduce_chunks_multi(sg, pl.nchunk, ntot, st);
        if (rc) return rc;
    }
    return GNAN_OK;
}
