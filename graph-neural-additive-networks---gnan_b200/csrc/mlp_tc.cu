// tcgen05 / TMEM path of the grouped shape-function MLPs (H = 64, 3 layers): the 64x64 hidden contraction runs on the
// 5th-generation tensor cores as a 3-term TF32 split (hi*hi + lo*hi + hi*lo, fp32 accumulation in TMEM), which keeps
// fp32-level accuracy (measured 1e-6 norm-wise by scratch/tc_probe.cu) at tensor-core speed.
//
// Reference lines replaced: GNAN.py:57-62,157 (forward), autograd through them (backward).
//
// Mapping (forward): a CTA owns two 128-row tiles ("groups"); a row thread owns one row = one TMEM lane.
//   layer 1: the row thread computes a[i] = relu(x*w1[i] + b1[i]) in registers, splits it into tf32 hi/lo and stores both
//            straight into TMEM with tcgen05.st (the A operand never touches shared memory);
//   layer 2: one elected thread issues tcgen05.mma kind::tf32 with A from TMEM and B = W2 (hi/lo, K-major core-matrix
//            layout) from shared memory, 8 K-steps x 3 terms, accumulating z[128x64] in TMEM; tcgen05.commit -> mbarrier;
//   layer 3: the row thread reads its z row back with tcgen05.ld, adds b2, ReLU, and contracts with wo in registers,
//            accumulating S[row, c] over the features of the chunk.
// Two producer warps stage the next feature's W2 split + small vectors into a double-buffered shared-memory slot while the
// current feature is consumed; the two row groups alternate so one group's CUDA-core work overlaps the other's MMAs.
#include <algorithm>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace {

constexpr int HID = 64;
constexpr int ROWS = 128;                 // rows per group (= TMEM lanes)
constexpr int FWD_GROUPS = 2;
constexpr int FWD_GROUP_THREADS = 256;    // 8 warps per group: 4 TMEM lane quadrants x 2 column halves (32 hidden units per thread)
constexpr int FWD_ROW_THREADS = FWD_GROUPS * FWD_GROUP_THREADS;
constexpr int PROD_THREADS = 64;
constexpr int FWD_ISSUE_THREADS = 32 * FWD_GROUPS;      // one MMA-issuer warp per group
constexpr int FWD_THREADS = FWD_ROW_THREADS + PROD_THREADS + FWD_ISSUE_THREADS;
constexpr int CT_MAX = 8;                 // output channels of the backward kernel and of the stacked (hi|lo along N) forward form
constexpr int CF_MAX = 64;                // output channels supported by the forward kernel (Y has 64 TMEM columns per group)

// Output-layer operand of the forward kernel, by padded channel count CP:
//   CP = 8 (C <= 8): ONE N = 16 MMA per K-step, rows n = c -> Wo_hi[c], n = 8 + c -> Wo_lo[c] (hi*hi and hi*lo in one instruction);
//   CP = 16/32/48/64: N = CP, separate hi and lo blocks, three MMA sets (a_hi Wo_hi + a_lo Wo_hi + a_hi Wo_lo) into the same Y.
template <int CP> struct YwCfg {
    static constexpr int N = CP <= 8 ? 16 : CP;            // N of the output-layer MMA (smallest legal N for M = 128 is 16)
    static constexpr int ROWS = CP <= 8 ? 16 : 2 * CP;     // operand rows held in the slot
    static constexpr int LO = CP <= 8 ? 8 * HID : CP * HID; // float offset of the lo rows (n-block 1 / the second block)
};

// shared-memory slot of one feature: B operands (hi/lo, UMMA K-major no-swizzle core-matrix layout) + small vectors
template <int CP>
struct __align__(16) FeatSlot {
    float bhi[HID * HID];                 // W2   [n=j][k=i]
    float blo[HID * HID];
    float yw[YwCfg<CP>::ROWS * HID];      // [n][k=j] (rows c >= C are zero)
    float w1[HID], b1[HID], b2[HID];
};

template <int CP>
struct FwdSmem {
    FeatSlot<CP> slot[2];
    float bo_sum[CF_MAX];                 // sum of the chunk's output biases
    uint64_t b_full[2], b_empty[2], a1_full[FWD_GROUPS], a2_full[FWD_GROUPS], d1_full[FWD_GROUPS], dy_full[FWD_GROUPS];
    uint32_t tmem_base;
};

struct TcArgs {
    const float *u;
    int64_t R, ldu;
    int G, C;
    const float *w1, *b1, *wh, *bh, *wo, *bo;
    uint32_t drop_thresh;
    float drop_scale;
    uint64_t seed;
    const uint64_t *seed_dev;   // optional device-resident seed word XORed into `seed` at kernel start (CUDA-graph replays)
    int single_pass;  // 1 = plain tf32 (no lo terms)
    const int64_t *grp_ptr;   // backward, entries mode (gnan_mlp_entries_bwd): rows of group g = its entries; NULL = dense
    // backward over a channel slice [c_off, c_off + C) of Ctot channels (C > 8 runs as ceil(C/8) passes whose gradients add up:
    // everything downstream of dh = sum_c g_c wo_c is linear in g); chunk_off = first partial-gradient slot of the pass
    int Ctot, c_off, chunk_off;
    // backward with the output layer outside the kernel (EXT: any C in ONE pass): dh_ext [R][G][HID] = dS Wo_g is read instead of
    // contracted here, a1_ext [R][G][HID] (the last hidden activation) is written for the caller's dWo GEMM
    const float *dh_ext;
    float *a1_ext;
};

__device__ __forceinline__ uint64_t tc_drop_key(const TcArgs &a, int layer, int g, int64_t row, int unit)
{
    return ((((uint64_t)layer * a.G + g) * (uint64_t)a.R + (uint64_t)row) * HID) + unit;   // same keys as the fp32 path
}

constexpr uint32_t B_LBO = 128, B_SBO = 2048, B_KSTEP = 256;   // bytes; one K-step = 8 tf32 = two 16-byte chunks

template <int CP>
__device__ __forceinline__ float produce_slot(FeatSlot<CP> &sl, const TcArgs &a, int g, int pt)
{
    const float *W = a.wh + (size_t)g * HID * HID;     // [j][i] = [n][k]
    float4 v[16];
#pragma unroll
    for (int t = 0; t < 16; ++t) {                      // all 16 loads in flight before the first use
        const int idx = pt + PROD_THREADS * t;          // 1024 float4 chunks: n fastest -> conflict-free 128-bit stores
        v[t] = __ldg(reinterpret_cast<const float4 *>(W + (idx & 63) * HID + (idx >> 6) * 4));
    }
#pragma unroll
    for (int t = 0; t < 16; ++t) {
        const int idx = pt + PROD_THREADS * t;
        const int n = idx & 63, kc = idx >> 6;
        uint32_t h0, h1, h2, h3, l0, l1, l2, l3;
        split_tf32(v[t].x, h0, l0); split_tf32(v[t].y, h1, l1); split_tf32(v[t].z, h2, l2); split_tf32(v[t].w, h3, l3);
        const int o = (n >> 3) * 512 + kc * 32 + (n & 7) * 4;
        *reinterpret_cast<uint4 *>(sl.bhi + o) = make_uint4(h0, h1, h2, h3);
        *reinterpret_cast<uint4 *>(sl.blo + o) = make_uint4(l0, l1, l2, l3);
    }
    sl.w1[pt] = __ldg(a.w1 + (size_t)g * HID + pt);
    sl.b1[pt] = a.b1 ? __ldg(a.b1 + (size_t)g * HID + pt) : 0.f;
    sl.b2[pt] = a.bh ? __ldg(a.bh + (size_t)g * HID + pt) : 0.f;
    // Wo[c][j = pt] -> K-major (n = c, k = j): (c/8)*512 + (j/4)*32 + (c%8)*4 + (j%4) floats
    for (int c = 0; c < a.C; ++c) {
        uint32_t h, l;
        split_tf32(__ldg(a.wo + ((size_t)g * a.C + c) * HID + pt), h, l);
        const int o = (c >> 3) * 512 + (pt >> 2) * 32 + (c & 7) * 4 + (pt & 3);      // hi rows first, lo rows YwCfg::LO floats later
        sl.yw[o] = __uint_as_float(h);
        sl.yw[YwCfg<CP>::LO + o] = __uint_as_float(l);
    }
    return (a.bo && pt < a.C) ? __ldg(a.bo + (size_t)g * a.C + pt) : 0.f;
}

// grid (row-pair tiles, feature chunks); Spart[chunk][R][C]
// Two 128-row groups per CTA; a row thread owns one row (TMEM lane) x 32 hidden units. Per feature and group:
//   gen   a0 = relu(x w1 + b1) -> TMEM A (hi|lo)                      | MMA1: z = a0 W2^T           (24 x M128 N64 K8)
//   epi   a1 = relu(z + b2)    -> TMEM A (hi|lo, overwriting a0)      | MMAy: Y += a1 Wo^T          (24 x M128 N16 K8)
// Y accumulates over the chunk's features in TMEM (the sum over groups f_k never leaves the tensor core) and is read once.
template <bool DROP, int CP>
__global__ void __launch_bounds__(FWD_THREADS, 1)
mlp_tc_fwd_kernel(TcArgs a, int KC, float *__restrict__ Spart)
{
    if (DROP && a.seed_dev) a.seed ^= *a.seed_dev;
    using YC = YwCfg<CP>;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    FwdSmem<CP> &sm = *reinterpret_cast<FwdSmem<CP> *>(smem_raw);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g0 = blockIdx.y * KC;
    const int ng = min(KC, a.G - g0);

    if (warp == 0) tmem_alloc(smem_u32(&sm.tmem_base), 512);
    if (tid == 32) {
        for (int s = 0; s < 2; ++s) {
            mbar_init(smem_u32(&sm.b_full[s]), PROD_THREADS);
            mbar_init(smem_u32(&sm.b_empty[s]), FWD_GROUPS);        // one tcgen05.commit per group
        }
        for (int gI = 0; gI < FWD_GROUPS; ++gI) {
            mbar_init(smem_u32(&sm.a1_full[gI]), FWD_GROUP_THREADS);
            mbar_init(smem_u32(&sm.a2_full[gI]), FWD_GROUP_THREADS);
            mbar_init(smem_u32(&sm.d1_full[gI]), 1);
            mbar_init(smem_u32(&sm.dy_full[gI]), 1);
        }
        mbar_init_fence();
    }
    if (tid >= FWD_ROW_THREADS && tid < FWD_ROW_THREADS + PROD_THREADS) {   // zero the output-layer operands once (rows c >= C stay zero)
        const int pt = tid - FWD_ROW_THREADS;
        for (int s = 0; s < 2; ++s)
            for (int i = pt; i < YC::ROWS * HID; i += PROD_THREADS) sm.slot[s].yw[i] = 0.f;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = sm.tmem_base;

    if (tid >= FWD_ROW_THREADS + PROD_THREADS) {
        // ===== MMA issuers: one warp per group =====
        const int grp = (tid - FWD_ROW_THREADS - PROD_THREADS) >> 5;
        const uint32_t gbase = tmem + (uint32_t)grp * 256;
        const uint32_t colA_hi = 0, colA_lo = 64, colD = 128, colY = 192;
        const uint32_t idesc = umma_idesc_tf32(128, 64), idesc_y = umma_idesc_tf32(128, YC::N);
        for (int kk = 0; kk < ng; ++kk) {
            const int s = kk & 1, n = kk >> 1;
            const FeatSlot<CP> &sl = sm.slot[s];
            mbar_wait(smem_u32(&sm.b_full[s]), n & 1);
            mbar_wait(smem_u32(&sm.a1_full[grp]), kk & 1);
            tc_fence_after();
            if (lane == 0) {
                const uint32_t bh = smem_u32(sl.bhi), bl = smem_u32(sl.blo);
#pragma unroll
                for (int ks = 0; ks < 8; ++ks)
                    umma_tf32_ts(gbase + colD, gbase + colA_hi + ks * 8, umma_desc_kmajor(bh + ks * B_KSTEP, B_LBO, B_SBO), idesc, ks > 0);
                if (!a.single_pass) {
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks)
                        umma_tf32_ts(gbase + colD, gbase + colA_lo + ks * 8, umma_desc_kmajor(bh + ks * B_KSTEP, B_LBO, B_SBO), idesc, 1);
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks)
                        umma_tf32_ts(gbase + colD, gbase + colA_hi + ks * 8, umma_desc_kmajor(bl + ks * B_KSTEP, B_LBO, B_SBO), idesc, 1);
                }
                umma_commit(smem_u32(&sm.d1_full[grp]));
            }
            __syncwarp();
            mbar_wait(smem_u32(&sm.a2_full[grp]), kk & 1);
            tc_fence_after();
            if (lane == 0) {
                // Y[:, c] += a1 Wo_hi[c], Y[:, 8+c] += a1 Wo_lo[c]: the hi|lo stacking along N gives hi*hi and hi*lo in one MMA
                const uint32_t yw = smem_u32(sl.yw);
#pragma unroll
                for (int ks = 0; ks < 8; ++ks)
                    umma_tf32_ts(gbase + colY, gbase + colA_hi + ks * 8, umma_desc_kmajor(yw + ks * B_KSTEP, B_LBO, B_SBO), idesc_y, (kk > 0 || ks > 0) ? 1u : 0u);
                if (!a.single_pass) {
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks)
                        umma_tf32_ts(gbase + colY, gbase + colA_lo + ks * 8, umma_desc_kmajor(yw + ks * B_KSTEP, B_LBO, B_SBO), idesc_y, 1);
                    if (CP > 8) {                            // the stacked form gets hi*lo from rows 8..15 of the same MMA
                        const uint32_t ywl = yw + (uint32_t)YC::LO * 4u;
#pragma unroll
                        for (int ks = 0; ks < 8; ++ks)
                            umma_tf32_ts(gbase + colY, gbase + colA_hi + ks * 8, umma_desc_kmajor(ywl + ks * B_KSTEP, B_LBO, B_SBO), idesc_y, 1);
                    }
                }
                umma_commit(smem_u32(&sm.dy_full[grp]));
                umma_commit(smem_u32(&sm.b_empty[s]));       // the slot is free once this group's MMAs on it are done
            }
            __syncwarp();
        }
    } else if (tid >= FWD_ROW_THREADS) {
        // ===== producers =====
        const int pt = tid - FWD_ROW_THREADS;
        float bsum = 0.f;
        for (int kk = 0; kk < ng; ++kk) {
            const int s = kk & 1, n = kk >> 1;
            mbar_wait(smem_u32(&sm.b_empty[s]), (n & 1) ^ 1);
            bsum += produce_slot(sm.slot[s], a, g0 + kk, pt);
            if (kk == ng - 1) sm.bo_sum[pt] = bsum;                  // PROD_THREADS == CF_MAX
            fence_async_smem();                      // make the generic-proxy writes visible to the tensor core
            mbar_arrive(smem_u32(&sm.b_full[s]));
        }
    } else {
        // ===== row threads =====
        const int grp = tid >> 8, wg = (tid >> 5) & 7;
        const int q = wg & 3, half = wg >> 2;
        const int rt = q * 32 + lane;                        // row inside the group's tile == TMEM lane
        const int c0 = half * 32;
        const int64_t row = ((int64_t)blockIdx.x * FWD_GROUPS + grp) * ROWS + rt;
        const bool row_ok = row < a.R;
        const uint32_t gbase = tmem + (uint32_t)grp * 256;   // this group's TMEM columns
        const uint32_t lane_base = gbase + ((uint32_t)(q * 32) << 16);
        const uint32_t colA_hi = 0, colA_lo = 64, colD = 128, colY = 192;
        float x_next = row_ok ? __ldg(a.u + row * a.ldu + g0) : 0.f;

        for (int kk = 0; kk < ng; ++kk) {
            const int s = kk & 1, n = kk >> 1, g = g0 + kk;
            const FeatSlot<CP> &sl = sm.slot[s];
            const float x = x_next;
            if (kk + 1 < ng && row_ok) x_next = ldg_prefetch(a.u + row * a.ldu + g + 1);
            mbar_wait(smem_u32(&sm.b_full[s]), n & 1);
            if (kk > 0) {                                   // A still holds a1 of the previous feature until its MMAy is done
                mbar_wait(smem_u32(&sm.dy_full[grp]), (kk - 1) & 1);
                tc_fence_after();
            }
            // ---- layer 1 -> TMEM (A operand, hi | lo), 16 units at a time
#pragma unroll
            for (int p = 0; p < 2; ++p) {
                uint32_t hi[16], lo[16];
#pragma unroll
                for (int i4 = 0; i4 < 4; ++i4) {
                    const float4 w = *reinterpret_cast<const float4 *>(sl.w1 + c0 + p * 16 + i4 * 4);
                    const float4 b = *reinterpret_cast<const float4 *>(sl.b1 + c0 + p * 16 + i4 * 4);
                    float v[4] = {fmaxf(fmaf(x, w.x, b.x), 0.f), fmaxf(fmaf(x, w.y, b.y), 0.f),
                                  fmaxf(fmaf(x, w.z, b.z), 0.f), fmaxf(fmaf(x, w.w, b.w), 0.f)};
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        if (DROP) v[e] *= gnan_dropout_mul(a.seed, tc_drop_key(a, 0, g, row, c0 + p * 16 + i4 * 4 + e), a.drop_thresh, a.drop_scale);
                        split_tf32(v[e], hi[i4 * 4 + e], lo[i4 * 4 + e]);
                    }
                }
                tmem_st16(lane_base + colA_hi + c0 + p * 16, hi);
                if (!a.single_pass) tmem_st16(lane_base + colA_lo + c0 + p * 16, lo);
            }
            tmem_wait_st();
            tc_fence_before();
            mbar_arrive(smem_u32(&sm.a1_full[grp]));             // the group's issuer warp runs MMA1
            mbar_wait(smem_u32(&sm.d1_full[grp]), kk & 1);
            tc_fence_after();
            // ---- a1 = relu(z + b2) -> TMEM A (MMA1 has consumed a0), 16 units at a time
#pragma unroll
            for (int p = 0; p < 2; ++p) {
                uint32_t d[16], hi[16], lo[16];
                tmem_ld16(lane_base + colD + c0 + p * 16, d);
                tmem_wait_ld();
#pragma unroll
                for (int j4 = 0; j4 < 4; ++j4) {
                    const float4 b = *reinterpret_cast<const float4 *>(sl.b2 + c0 + p * 16 + j4 * 4);
                    float h[4] = {fmaxf(__uint_as_float(d[j4 * 4 + 0]) + b.x, 0.f), fmaxf(__uint_as_float(d[j4 * 4 + 1]) + b.y, 0.f),
                                  fmaxf(__uint_as_float(d[j4 * 4 + 2]) + b.z, 0.f), fmaxf(__uint_as_float(d[j4 * 4 + 3]) + b.w, 0.f)};
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        if (DROP) h[e] *= gnan_dropout_mul(a.seed, tc_drop_key(a, 1, g, row, c0 + p * 16 + j4 * 4 + e), a.drop_thresh, a.drop_scale);
                        split_tf32(h[e], hi[j4 * 4 + e], lo[j4 * 4 + e]);
                    }
                }
                tmem_st16(lane_base + colA_hi + c0 + p * 16, hi);
                if (!a.single_pass) tmem_st16(lane_base + colA_lo + c0 + p * 16, lo);
            }
            tmem_wait_st();
            tc_fence_before();
            mbar_arrive(smem_u32(&sm.a2_full[grp]));             // the group's issuer warp runs the output-layer MMAs
        }
        // ---- S[row, c] = Y + sum of output biases
        mbar_wait(smem_u32(&sm.dy_full[grp]), (ng - 1) & 1);
        tc_fence_after();
        if (CP <= 8) {
            if (half == 0) {
                uint32_t y[16];
                tmem_ld16(lane_base + colY, y);
                tmem_wait_ld();
                if (row_ok) {
                    float *out = Spart + ((size_t)blockIdx.y * a.R + row) * a.C;
#pragma unroll
                    for (int c = 0; c < CT_MAX; ++c)
                        if (c < a.C) out[c] = (__uint_as_float(y[c]) + __uint_as_float(y[8 + c])) + sm.bo_sum[c];
                }
            }
        } else {
            // 16-column chunks of Y alternate between the two column halves of the quadrant's warps
#pragma unroll
            for (int n0 = 0; n0 < CP; n0 += 16) {
                if (((n0 >> 4) & 1) != half) continue;
                uint32_t y[16];
                tmem_ld16(lane_base + colY + n0, y);
                tmem_wait_ld();
                if (row_ok) {
                    float *out = Spart + ((size_t)blockIdx.y * a.R + row) * a.C;
#pragma unroll
                    for (int c = 0; c < 16; ++c)
                        if (n0 + c < a.C) out[n0 + c] = __uint_as_float(y[c]) + sm.bo_sum[n0 + c];
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

// ---- forward, entries mode (gnan_mlp_entries_fwd_ex) ----------------------------------------------------------------------
// Y[e,:] = f_g(val[e]) per entry (no sum over groups: gnan_entries_to_rows does that). A work item = (group, 128-entry tile of
// that group). The CTA is persistent; its two row groups consume DIFFERENT items (item 2i and 2i+1 of the CTA's stride), so each
// row group has its own double-buffered weight slot, its own 64 producer threads and its own MMA-issuer warp; the pipeline per
// item is the dense forward's (layer 1 -> TMEM, MMA1, a1 -> TMEM, output-layer MMA with hi|lo stacked along N), except that Y
// starts from zero at every item and is read back one item later (while that item's layer 1 is generated). No dropout.
constexpr int ENT_PROD_THREADS = FWD_GROUPS * PROD_THREADS;
constexpr int ENT_THREADS = FWD_ROW_THREADS + ENT_PROD_THREADS + FWD_ISSUE_THREADS;

struct EntSmem {
    FeatSlot<8> slot[FWD_GROUPS][2];
    uint64_t b_full[FWD_GROUPS][2], b_empty[FWD_GROUPS][2], a1_full[FWD_GROUPS], a2_full[FWD_GROUPS], d1_full[FWD_GROUPS], dy_full[FWD_GROUPS];
    uint32_t tmem_base;
};

__global__ void __launch_bounds__(ENT_THREADS, 1)
mlp_tc_entries_fwd_kernel(TcArgs a, const int32_t *__restrict__ items, int64_t n_items, float *__restrict__ Y)
{
    using YC = YwCfg<8>;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    EntSmem &sm = *reinterpret_cast<EntSmem *>(smem_raw);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t stride = (int64_t)gridDim.x * FWD_GROUPS;

    if (warp == 0) tmem_alloc(smem_u32(&sm.tmem_base), 512);
    if (tid == 32) {
        for (int gI = 0; gI < FWD_GROUPS; ++gI) {
            for (int s2 = 0; s2 < 2; ++s2) {
                mbar_init(smem_u32(&sm.b_full[gI][s2]), PROD_THREADS);
                mbar_init(smem_u32(&sm.b_empty[gI][s2]), 1);
            }
            mbar_init(smem_u32(&sm.a1_full[gI]), FWD_GROUP_THREADS);
            mbar_init(smem_u32(&sm.a2_full[gI]), FWD_GROUP_THREADS);
            mbar_init(smem_u32(&sm.d1_full[gI]), 1);
            mbar_init(smem_u32(&sm.dy_full[gI]), 1);
        }
        mbar_init_fence();
    }
    if (tid >= FWD_ROW_THREADS && tid < FWD_ROW_THREADS + ENT_PROD_THREADS) {   // output-layer operand rows c >= C stay zero
        const int pq = tid - FWD_ROW_THREADS;
        for (int gI = 0; gI < FWD_GROUPS; ++gI)
            for (int s2 = 0; s2 < 2; ++s2)
                for (int i = pq; i < YC::ROWS * HID; i += ENT_PROD_THREADS) sm.slot[gI][s2].yw[i] = 0.f;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = sm.tmem_base;

    if (tid >= FWD_ROW_THREADS + ENT_PROD_THREADS) {
        // ===== MMA issuers: one warp per row group =====
        const int grp = (tid - FWD_ROW_THREADS - ENT_PROD_THREADS) >> 5;
        const uint32_t gbase = tmem + (uint32_t)grp * 256;
        const uint32_t colA_hi = 0, colA_lo = 64, colD = 128, colY = 192;
        const uint32_t idesc = umma_idesc_tf32(128, 64), idesc_y = umma_idesc_tf32(128, YC::N);
        int kk = 0;
        for (int64_t it = (int64_t)blockIdx.x * FWD_GROUPS + grp; it < n_items; it += stride, ++kk) {
            const int s = kk & 1, n = kk >> 1;
            const FeatSlot<8> &sl = sm.slot[grp][s];
            mbar_wait(smem_u32(&sm.b_full[grp][s]), n & 1);
            mbar_wait(smem_u32(&sm.a1_full[grp]), kk & 1);
            tc_fence_after();
            if (lane == 0) {
                const uint32_t bh = smem_u32(sl.bhi), bl = smem_u32(sl.blo);
#pragma unroll
                for (int ks = 0; ks < 8; ++ks)
                    umma_tf32_ts(gbase + colD, gbase + colA_hi + ks * 8, umma_desc_kmajor(bh + ks * B_KSTEP, B_LBO, B_SBO), idesc, ks > 0);
                if (!a.single_pass) {
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks)
                        umma_tf32_ts(gbase + colD, gbase + colA_lo + ks * 8, umma_desc_kmajor(bh + ks * B_KSTEP, B_LBO, B_SBO), idesc, 1);
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks)
                        umma_tf32_ts(gbase + colD, gbase + colA_hi + ks * 8, umma_desc_kmajor(bl + ks * B_KSTEP, B_LBO, B_SBO), idesc, 1);
                }
                umma_commit(smem_u32(&sm.d1_full[grp]));
            }
            __syncwarp();
            mbar_wait(smem_u32(&sm.a2_full[grp]), kk & 1);
            tc_fence_after();
            if (lane == 0) {
                const uint32_t yw = smem_u32(sl.yw);
#pragma unroll
                for (int ks = 0; ks < 8; ++ks)
                    umma_tf32_ts(gbase + colY, gbase + colA_hi + ks * 8, umma_desc_kmajor(yw + ks * B_KSTEP, B_LBO, B_SBO), idesc_y, ks > 0 ? 1u : 0u);
                if (!a.single_pass) {
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks)
                        umma_tf32_ts(gbase + colY, gbase + colA_lo + ks * 8, umma_desc_kmajor(yw + ks * B_KSTEP, B_LBO, B_SBO), idesc_y, 1);
                }
                umma_commit(smem_u32(&sm.dy_full[grp]));
                umma_commit(smem_u32(&sm.b_empty[grp][s]));
            }
            __syncwarp();
        }
    } else if (tid >= FWD_ROW_THREADS) {
        // ===== producers: 64 threads per row group =====
        const int pq = tid - FWD_ROW_THREADS, grp = pq >> 6, pt = pq & 63;
        int kk = 0;
        for (int64_t it = (int64_t)blockIdx.x * FWD_GROUPS + grp; it < n_items; it += stride, ++kk) {
            const int s = kk & 1, n = kk >> 1;
            const int g = __ldg(items + 2 * it);
            mbar_wait(smem_u32(&sm.b_empty[grp][s]), (n & 1) ^ 1);
            (void)produce_slot<8>(sm.slot[grp][s], a, g, pt);
            fence_async_smem();
            mbar_arrive(smem_u32(&sm.b_full[grp][s]));
        }
    } else {
        // ===== row threads =====
        const int grp = tid >> 8, wg = (tid >> 5) & 7;
        const int q = wg & 3, half = wg >> 2;
        const int rt = q * 32 + lane;
        const int c0 = half * 32;
        const uint32_t gbase = tmem + (uint32_t)grp * 256;
        const uint32_t lane_base = gbase + ((uint32_t)(q * 32) << 16);
        const uint32_t colA_hi = 0, colA_lo = 64, colD = 128, colY = 192;
        // the item after the current one is resolved one iteration ahead (items -> grp_ptr -> val is a dependent load chain)
        auto resolve = [&](int64_t it, int64_t &erow, float &x, int &g) {
            erow = -1; x = 0.f; g = 0;
            if (it < n_items) {
                g = __ldg(items + 2 * it);
                const int tile = __ldg(items + 2 * it + 1);
                const int64_t eb = __ldg(a.grp_ptr + g), ne = __ldg(a.grp_ptr + g + 1) - eb;
                const int64_t r = (int64_t)tile * ROWS + rt;
                if (r < ne) { erow = eb + r; x = __ldg(a.u + erow); }
            }
        };
        int64_t it = (int64_t)blockIdx.x * FWD_GROUPS + grp;
        int64_t erow_n, erow_p = -1;
        float x_n, bo_p[CT_MAX];
        int g_n;
        resolve(it, erow_n, x_n, g_n);
        int kk = 0;
        auto write_prev = [&]() {           // Y of the previous item (its output-layer MMAs are complete)
            if (half == 0) {
                uint32_t y[16];
                tmem_ld16(lane_base + colY, y);
                tmem_wait_ld();
                if (erow_p >= 0) {
                    float *out = Y + erow_p * a.C;
#pragma unroll
                    for (int c = 0; c < CT_MAX; ++c)
                        if (c < a.C) out[c] = (__uint_as_float(y[c]) + __uint_as_float(y[8 + c])) + bo_p[c];
                }
            }
        };
        for (; it < n_items; it += stride, ++kk) {
            const int s = kk & 1, n = kk >> 1;
            const FeatSlot<8> &sl = sm.slot[grp][s];
            const float x = x_n;
            const int64_t erow = erow_n;
            const int g = g_n;
            mbar_wait(smem_u32(&sm.b_full[grp][s]), n & 1);
            if (kk > 0) {
                mbar_wait(smem_u32(&sm.dy_full[grp]), (kk - 1) & 1);
                tc_fence_after();
                write_prev();
                tc_fence_before();
            }
            erow_p = erow;
            if (half == 0) {
#pragma unroll
                for (int c = 0; c < CT_MAX; ++c) bo_p[c] = (a.bo && c < a.C) ? __ldg(a.bo + (size_t)g * a.C + c) : 0.f;
            }
#pragma unroll
            for (int p = 0; p < 2; ++p) {
                uint32_t hi[16], lo[16];
#pragma unroll
                for (int i4 = 0; i4 < 4; ++i4) {
                    const float4 w = *reinterpret_cast<const float4 *>(sl.w1 + c0 + p * 16 + i4 * 4);
                    const float4 b = *reinterpret_cast<const float4 *>(sl.b1 + c0 + p * 16 + i4 * 4);
                    const float v[4] = {fmaxf(fmaf(x, w.x, b.x), 0.f), fmaxf(fmaf(x, w.y, b.y), 0.f),
                                        fmaxf(fmaf(x, w.z, b.z), 0.f), fmaxf(fmaf(x, w.w, b.w), 0.f)};
#pragma unroll
                    for (int e = 0; e < 4; ++e) split_tf32(v[e], hi[i4 * 4 + e], lo[i4 * 4 + e]);
                }
                tmem_st16(lane_base + colA_hi + c0 + p * 16, hi);
                if (!a.single_pass) tmem_st16(lane_base + colA_lo + c0 + p * 16, lo);
            }
            tmem_wait_st();
            tc_fence_before();
            mbar_arrive(smem_u32(&sm.a1_full[grp]));
            resolve(it + stride, erow_n, x_n, g_n);            // under MMA1
            mbar_wait(smem_u32(&sm.d1_full[grp]), kk & 1);
            tc_fence_after();
#pragma unroll
            for (int p = 0; p < 2; ++p) {
                uint32_t d[16], hi[16], lo[16];
                tmem_ld16(lane_base + colD + c0 + p * 16, d);
                tmem_wait_ld();
#pragma unroll
                for (int j4 = 0; j4 < 4; ++j4) {
                    const float4 b = *reinterpret_cast<const float4 *>(sl.b2 + c0 + p * 16 + j4 * 4);
                    const float h[4] = {fmaxf(__uint_as_float(d[j4 * 4 + 0]) + b.x, 0.f), fmaxf(__uint_as_float(d[j4 * 4 + 1]) + b.y, 0.f),
                                        fmaxf(__uint_as_float(d[j4 * 4 + 2]) + b.z, 0.f), fmaxf(__uint_as_float(d[j4 * 4 + 3]) + b.w, 0.f)};
#pragma unroll
                    for (int e = 0; e < 4; ++e) split_tf32(h[e], hi[j4 * 4 + e], lo[j4 * 4 + e]);
                }
                tmem_st16(lane_base + colA_hi + c0 + p * 16, hi);
                if (!a.single_pass) tmem_st16(lane_base + colA_lo + c0 + p * 16, lo);
            }
            tmem_wait_st();
            tc_fence_before();
            mbar_arrive(smem_u32(&sm.a2_full[grp]));
        }
        if (kk > 0) {
            mbar_wait(smem_u32(&sm.dy_full[grp]), (kk - 1) & 1);
            tc_fence_after();
            write_prev();
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

// ---- backward ---------------------------------------------------------------------------------------------------------
// CTA <-> (feature g, row chunk), 16 row warps + 1 MMA warp. A row warp owns 32 rows (one TMEM lane quadrant) x 16 of the
// 64 hidden units (warps w, w+4, w+8, w+12 share a quadrant). In entries mode (TcArgs::grp_ptr) the rows are the group's own
// entries instead of column g of the dense matrix. Per 128-row tile:
//   gen    a0 = relu(x w1 + b1) -> TMEM A (hi|lo)  and  -> smem sH (K-major over rows: B operand of MMA3)
//   MMA1   z2 = a0 W2^T                                    (TS, 24 x [128x64x8])
//   epiC   a1 = relu(z2+b2); dz2 = (g Wo) * 1[a1>0] -> TMEM A (hi|lo) and -> smem sZ (A operand of MMA3); db2 partial sums
//   MMA2   d1 = dz2 W2                                     (TS, B = W2^T copy, 24 MMAs)
//   MMA3   dW2 += [dz2_hi | dz2_lo]^T [a0_hi ; a0_lo]      (SS, M = 128 stacks hi/lo: all four split terms, 32 MMAs,
//                                                           accumulator persistent in TMEM across the CTA's tiles)
//   epiF   dz1 = d1 * 1[a0>0]; dw1/db1 partial sums
//   dWo    a1 recomputed from TMEM, staged to smem (reusing sZ once MMA3 is done), dWo[c][j] += g[r][c] a1[r][j]
// All smem operands are K-major with LBO = 144 B (a 16-byte skew per K chunk makes the transposing 4-byte stores of a
// warp bank-conflict free); MN-major tf32 descriptors returned zeros on B200 (scratch/tc_probe3.cu), so they are avoided.
constexpr int BWD_NS = 4;                           // column split: a TMEM lane quadrant is shared by NS warps, 64/NS units each
constexpr int BWD_COLS = HID / BWD_NS;              // hidden units per row thread
constexpr int BWD_ROW_WARPS = 4 * BWD_NS;
constexpr int BWD_ROW_THREADS = 32 * BWD_ROW_WARPS;
constexpr int BWD_THREADS = BWD_ROW_THREADS + 32;
constexpr uint32_t T_LBO = 144;                    // bytes between K chunks (4 rows) of a transposed operand
constexpr uint32_t T_SBO = 32 * T_LBO;             // 128 rows = 32 chunks per 8-unit block: 4608 B
constexpr uint32_t T_KSTEP = 2 * T_LBO;            // one MMA K-step = 8 rows
constexpr int T_BLK_FLOATS = T_SBO / 4;            // 1152 floats per 8-unit block

struct BwdSmem {
    float w_hi[HID * HID], w_lo[HID * HID];        // W2   [n=j][k=i]  (MMA1 B)
    float wt_hi[HID * HID], wt_lo[HID * HID];      // W2^T [n=i][k=j]  (MMA2 B)
    float sZ[16 * T_BLK_FLOATS];                   // dz2^T: 16 blocks of 8 units: 0-7 = hi, 8-15 = lo  (MMA3 A, M = 128); later scratch
    float sH_hi[8 * T_BLK_FLOATS];                 // a0^T hi (MMA3 B, N = 64)
    float sH_lo[8 * T_BLK_FLOATS];
    float w1[HID], b1[HID], b2[HID];
    float wok_hi[HID * CT_MAX], wok_lo[HID * CT_MAX];  // Wo^T as a K-major B operand [n=j][k=c] (K = 8): dh = g Wo on the tensor core
    float sG[2][ROWS][CT_MAX];                     // dS tile, double-buffered by tile parity (read one tile later by the dWo phase)
    float red[BWD_ROW_WARPS][2 * BWD_COLS];        // cross-warp staging for the small reductions
    uint64_t a1_full, a2_full, a3_full, d1_full, d2_full, d3_full;
    uint32_t tmem_base;
};

// float offset of (unit, row) inside a transposed K-major operand (unit = M/N index, row = K index)
__device__ __forceinline__ int tidx(int unit, int row) { return (unit >> 3) * T_BLK_FLOATS + (row >> 2) * 36 + (unit & 7) * 4 + (row & 3); }

// column sums over the 32 rows of a warp for N = 32 or 16 columns held as v[N]: on return every lane holds the sum of
// column (lane & (N-1))
template <int N>
__device__ __forceinline__ float warp_colsum(float (&v)[N], int lane)
{
#pragma unroll
    for (int w = N / 2; w >= 1; w >>= 1) {
        const bool up = (lane & w) != 0;
#pragma unroll
        for (int i = 0; i < w; ++i) {
            const float send = up ? v[i] : v[i + w];
            const float keep = up ? v[i + w] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, w);
        }
    }
    float r = v[0];
#pragma unroll
    for (int w = N; w < 32; w <<= 1) r += __shfl_xor_sync(0xffffffffu, r, w);
    return r;
}

template <int N> struct TmemIO;
template <> struct TmemIO<32> {
    static __device__ __forceinline__ void st(uint32_t t, const uint32_t (&v)[32]) { tmem_st32(t, v); }
    static __device__ __forceinline__ void ld(uint32_t t, uint32_t (&v)[32]) { tmem_ld32(t, v); }
};
template <> struct TmemIO<16> {
    static __device__ __forceinline__ void st(uint32_t t, const uint32_t (&v)[16]) { tmem_st16(t, v); }
    static __device__ __forceinline__ void ld(uint32_t t, uint32_t (&v)[16]) { tmem_ld16(t, v); }
};

struct TcGradPtrs { float *w1, *b1, *wh, *bh, *wo, *bo; size_t chunk_stride; };

template <int CT, bool DROP, bool EXT = false>
__global__ void __launch_bounds__(BWD_THREADS, 1)   // 17 warps occupy 20 warp slots (5 per scheduler): 96 registers is the cap
mlp_tc_bwd_kernel(TcArgs a, const float *__restrict__ dS, TcGradPtrs gp, int64_t ntiles)
{
    if (DROP && a.seed_dev) a.seed ^= *a.seed_dev;
    constexpr int NC = BWD_COLS;
    using IO = TmemIO<NC>;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    BwdSmem &sm = *reinterpret_cast<BwdSmem *>(smem_raw);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = blockIdx.y;
    // row space of this CTA's group: all R rows, column g of u (dense), or the group's own entries (entries mode)
    int64_t nrow = a.R, ustride = a.ldu;
    const float *ub = a.u + g;
    if (a.grp_ptr) {
        const int64_t ebase = a.grp_ptr[g];
        nrow = a.grp_ptr[g + 1] - ebase;
        ntiles = (nrow + ROWS - 1) / ROWS;
        ub = a.u + ebase;
        ustride = 1;
        dS += ebase * a.Ctot;
    }
    dS += a.c_off;

    if (warp == BWD_ROW_WARPS) tmem_alloc(smem_u32(&sm.tmem_base), 512);
    if (tid == 0) {
        mbar_init(smem_u32(&sm.a1_full), BWD_ROW_THREADS);
        mbar_init(smem_u32(&sm.a2_full), BWD_ROW_THREADS);
        mbar_init(smem_u32(&sm.a3_full), BWD_ROW_THREADS);
        mbar_init(smem_u32(&sm.d1_full), 1);
        mbar_init(smem_u32(&sm.d2_full), 1);
        mbar_init(smem_u32(&sm.d3_full), 1);
        mbar_init_fence();
    }
    // stage the feature's weights: W2 and W2^T split into hi/lo in the K-major core-matrix layout (LBO 128, SBO 2048)
    {
        const float *W = a.wh + (size_t)g * HID * HID;
        for (int idx = tid; idx < HID * HID; idx += BWD_THREADS) {
            const int j = idx >> 6, i = idx & 63;
            uint32_t h, l;
            split_tf32(__ldg(W + idx), h, l);
            const int o = (j >> 3) * 512 + (i >> 2) * 32 + (j & 7) * 4 + (i & 3);       // (n=j, k=i)
            const int ot = (i >> 3) * 512 + (j >> 2) * 32 + (i & 7) * 4 + (j & 3);      // (n=i, k=j)
            sm.w_hi[o] = __uint_as_float(h); sm.w_lo[o] = __uint_as_float(l);
            sm.wt_hi[ot] = __uint_as_float(h); sm.wt_lo[ot] = __uint_as_float(l);
        }
        if (tid < HID) {
            sm.w1[tid] = __ldg(a.w1 + (size_t)g * HID + tid);
            sm.b1[tid] = a.b1 ? __ldg(a.b1 + (size_t)g * HID + tid) : 0.f;
            sm.b2[tid] = a.bh ? __ldg(a.bh + (size_t)g * HID + tid) : 0.f;
            for (int c = 0; c < CT_MAX; ++c) {
                const float v = c < a.C ? __ldg(a.wo + ((size_t)g * a.Ctot + a.c_off + c) * HID + tid) : 0.f;
                uint32_t h, l;
                split_tf32(v, h, l);
                const int o = (tid >> 3) * 64 + (c >> 2) * 32 + (tid & 7) * 4 + (c & 3);   // (n=tid, k=c): LBO 128 B, SBO 256 B
                sm.wok_hi[o] = __uint_as_float(h); sm.wok_lo[o] = __uint_as_float(l);
            }
        }
        // the 16-byte gaps between K chunks are never read; zero the operand buffers once anyway (no NaN garbage)
        for (int idx = tid; idx < 16 * T_BLK_FLOATS; idx += BWD_THREADS) sm.sZ[idx] = 0.f;
        for (int idx = tid; idx < 8 * T_BLK_FLOATS; idx += BWD_THREADS) { sm.sH_hi[idx] = 0.f; sm.sH_lo[idx] = 0.f; }
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = sm.tmem_base;
    const uint32_t colA_hi = 0, colA_lo = 64, colD1 = 128, colD2 = 192, colD3 = 256, colG_hi = 320, colG_lo = 328, colDH = 336, colD1b = 400;   // D1 is double-buffered (D1 / D1b by tile parity)

    if (warp == BWD_ROW_WARPS) {
        // ===== MMA issuer =====
        const uint32_t idesc = umma_idesc_tf32(128, 64);
        uint32_t it = 0;
        for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++it) {
            const uint32_t ph = it & 1;
            mbar_wait(smem_u32(&sm.a1_full), ph);
            tc_fence_after();
            if (lane == 0) {
                const uint32_t bh = smem_u32(sm.w_hi), bl = smem_u32(sm.w_lo);
                const uint32_t d1 = tmem + (ph ? colD1b : colD1);
#pragma unroll
                for (int ks = 0; ks < 8; ++ks)
                    umma_tf32_ts(d1, tmem + colA_hi + ks * 8, umma_desc_kmajor(bh + ks * B_KSTEP, B_LBO, B_SBO), idesc, ks > 0);
                if (!a.single_pass) {
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks)
                        umma_tf32_ts(d1, tmem + colA_lo + ks * 8, umma_desc_kmajor(bh + ks * B_KSTEP, B_LBO, B_SBO), idesc, 1);
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks)
                        umma_tf32_ts(d1, tmem + colA_hi + ks * 8, umma_desc_kmajor(bl + ks * B_KSTEP, B_LBO, B_SBO), idesc, 1);
                }
                // dh[r][j] = sum_c g[r][c] wo[c][j]: one K-step (K = 8 channels) per split term (EXT: dh comes from global memory)
                if (!EXT) {
                    const uint32_t wkh = smem_u32(sm.wok_hi), wkl = smem_u32(sm.wok_lo);
                    umma_tf32_ts(tmem + colDH, tmem + colG_hi, umma_desc_kmajor(wkh, 128, 256), idesc, 0);
                    if (!a.single_pass) {
                        umma_tf32_ts(tmem + colDH, tmem + colG_lo, umma_desc_kmajor(wkh, 128, 256), idesc, 1);
                        umma_tf32_ts(tmem + colDH, tmem + colG_hi, umma_desc_kmajor(wkl, 128, 256), idesc, 1);
                    }
                }
                umma_commit(smem_u32(&sm.d1_full));
            }
            __syncwarp();
            mbar_wait(smem_u32(&sm.a2_full), ph);
            tc_fence_after();
            if (lane == 0) {
                const uint32_t bh = smem_u32(sm.wt_hi), bl = smem_u32(sm.wt_lo);
#pragma unroll
                for (int ks = 0; ks < 8; ++ks)
                    umma_tf32_ts(tmem + colD2, tmem + colA_hi + ks * 8, umma_desc_kmajor(bh + ks * B_KSTEP, B_LBO, B_SBO), idesc, ks > 0);
                if (!a.single_pass) {
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks)
                        umma_tf32_ts(tmem + colD2, tmem + colA_lo + ks * 8, umma_desc_kmajor(bh + ks * B_KSTEP, B_LBO, B_SBO), idesc, 1);
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks)
                        umma_tf32_ts(tmem + colD2, tmem + colA_hi + ks * 8, umma_desc_kmajor(bl + ks * B_KSTEP, B_LBO, B_SBO), idesc, 1);
                }
                umma_commit(smem_u32(&sm.d2_full));
            }
            __syncwarp();
            mbar_wait(smem_u32(&sm.a3_full), ph);      // the transposed smem operands of MMA3 are staged off the MMA2 critical path
            tc_fence_after();
            if (lane == 0) {
                // dW2 accumulation over the 128 rows of the tile: A = sZ (M = 128: hi|lo), B = sH hi then lo
                const uint32_t za = smem_u32(sm.sZ), hh = smem_u32(sm.sH_hi), hl = smem_u32(sm.sH_lo);
#pragma unroll 4
                for (int ks = 0; ks < 16; ++ks)
                    umma_tf32_ss(tmem + colD3, umma_desc_kmajor(za + ks * T_KSTEP, T_LBO, T_SBO),
                                 umma_desc_kmajor(hh + ks * T_KSTEP, T_LBO, T_SBO), idesc, (it > 0 || ks > 0) ? 1u : 0u);
                if (!a.single_pass) {
#pragma unroll 4
                    for (int ks = 0; ks < 16; ++ks)
                        umma_tf32_ss(tmem + colD3, umma_desc_kmajor(za + ks * T_KSTEP, T_LBO, T_SBO),
                                     umma_desc_kmajor(hl + ks * T_KSTEP, T_LBO, T_SBO), idesc, 1);
                }
                umma_commit(smem_u32(&sm.d3_full));
            }
            __syncwarp();
        }
    } else {
        // ===== row warps =====
        const int q = warp & 3, part = warp >> 2;          // TMEM lane quadrant, column part
        const int r = q * 32 + lane;                       // row inside the tile == TMEM lane
        const int c0 = part * NC;                          // this thread's NC hidden units
        const uint32_t lane_base = tmem + ((uint32_t)(q * 32) << 16);
        constexpr int DWO_ROWS = ROWS / (BWD_ROW_THREADS / 64);   // rows per thread in the dWo loop
        float acc_wo[CT];                                  // dWo[c][j = tid & 63] over rows (tid >> 6)*DWO_ROWS.. of every tile
#pragma unroll
        for (int c = 0; c < CT; ++c) acc_wo[c] = 0.f;
        float p_b2 = 0.f, p_b1 = 0.f, p_w1 = 0.f;          // column (c0 + (lane & (NC-1))) sums over this warp's rows
        uint32_t it = 0;
        // x and dS of the next tile are fetched one tile ahead (their ~700-cycle latency was exposed in the gen phase)
        float x_n = 0.f, gv_n[CT];
        {
            const int64_t row = (int64_t)blockIdx.x * ROWS + r;
            const bool ok = blockIdx.x < ntiles && row < nrow;
            x_n = ok ? __ldg(ub + row * ustride) : 0.f;
#pragma unroll
            for (int c = 0; c < CT; ++c) gv_n[c] = (!EXT && ok && c < a.C && part == 0) ? __ldg(dS + row * a.Ctot + c) : 0.f;
        }
        // dWo phase of tile `tp` (parity php): a1 recomputed from D1[php], staged to the scratch tile (sZ, free once MMA3 of
        // that tile is done), dWo[c][j] += g[r][c] a1[r][j]. Runs while the tensor core works on the NEXT tile's MMA1.
        auto dwo_phase = [&](int64_t tp, uint32_t php) {      // caller has waited d3_full of that tile
            const int64_t rowp = tp * ROWS + r;
            uint32_t d[NC];
            IO::ld(lane_base + (php ? colD1b : colD1) + c0, d);
            tmem_wait_ld();
            float *scr = sm.sZ;
#pragma unroll
            for (int j4 = 0; j4 < NC / 4; ++j4) {
                const float4 b = *reinterpret_cast<const float4 *>(sm.b2 + c0 + j4 * 4);
                float v[4] = {fmaxf(__uint_as_float(d[j4 * 4 + 0]) + b.x, 0.f), fmaxf(__uint_as_float(d[j4 * 4 + 1]) + b.y, 0.f),
                              fmaxf(__uint_as_float(d[j4 * 4 + 2]) + b.z, 0.f), fmaxf(__uint_as_float(d[j4 * 4 + 3]) + b.w, 0.f)};
                if (DROP) {
#pragma unroll
                    for (int e = 0; e < 4; ++e)
                        v[e] *= gnan_dropout_mul(a.seed, tc_drop_key(a, 1, g, rowp, c0 + j4 * 4 + e), a.drop_thresh, a.drop_scale);
                }
                *reinterpret_cast<float4 *>(scr + r * 68 + c0 + j4 * 4) = make_float4(v[0], v[1], v[2], v[3]);
            }
            tc_fence_before();
            named_bar_sync(1, BWD_ROW_THREADS);
            const int j = tid & 63, r0 = (tid >> 6) * DWO_ROWS;
#pragma unroll 4
            for (int rr = 0; rr < DWO_ROWS; ++rr) {
                const float hv = scr[(r0 + rr) * 68 + j];
                const float4 g0 = *reinterpret_cast<const float4 *>(&sm.sG[php][r0 + rr][0]);
                const float4 g1 = *reinterpret_cast<const float4 *>(&sm.sG[php][r0 + rr][4]);
                const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
                for (int c = 0; c < CT; ++c) acc_wo[c] = fmaf(gg[c], hv, acc_wo[c]);
            }
            named_bar_sync(1, BWD_ROW_THREADS);          // the scratch tile is rewritten (as sZ) by the current tile's epiC
        };

        for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++it) {
            const uint32_t ph = it & 1;
            const int64_t row = t * ROWS + r;
            const float x = x_n;
            const int64_t tn = t + gridDim.x, rown = tn * ROWS + r;
            const bool okn = tn < ntiles && rown < nrow;
            x_n = 0.f;
            if (okn) x_n = ldg_prefetch(ub + rown * ustride);
            if (!EXT && part == 0) {                           // only these threads need dS: stage it for the dh MMA and the dWo phase
                uint32_t gh[CT_MAX], gl[CT_MAX];
#pragma unroll
                for (int c = 0; c < CT_MAX; ++c) {
                    const float v = c < CT ? gv_n[c < CT ? c : 0] : 0.f;
                    sm.sG[ph][r][c] = v;
                    split_tf32(v, gh[c], gl[c]);
                }
                tmem_st8(lane_base + colG_hi, gh);
                tmem_st8(lane_base + colG_lo, gl);
#pragma unroll
                for (int c = 0; c < CT; ++c) {
                    gv_n[c] = 0.f;
                    if (okn && c < a.C) gv_n[c] = ldg_prefetch(dS + rown * a.Ctot + c);
                }
            }
            // ---- [A] gen: a0 for units c0..c0+NC-1 -> TMEM only (the A operand of MMA1); then release the tensor core
            uint32_t hi[NC], lo[NC];
#pragma unroll
            for (int i4 = 0; i4 < NC / 4; ++i4) {
                const float4 w = *reinterpret_cast<const float4 *>(sm.w1 + c0 + i4 * 4);
                const float4 b = *reinterpret_cast<const float4 *>(sm.b1 + c0 + i4 * 4);
                float v[4] = {fmaxf(fmaf(x, w.x, b.x), 0.f), fmaxf(fmaf(x, w.y, b.y), 0.f),
                              fmaxf(fmaf(x, w.z, b.z), 0.f), fmaxf(fmaf(x, w.w, b.w), 0.f)};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    if (DROP) v[e] *= gnan_dropout_mul(a.seed, tc_drop_key(a, 0, g, row, c0 + i4 * 4 + e), a.drop_thresh, a.drop_scale);
                    split_tf32(v[e], hi[i4 * 4 + e], lo[i4 * 4 + e]);
                }
            }
            IO::st(lane_base + colA_hi + c0, hi);
            if (!a.single_pass) IO::st(lane_base + colA_lo + c0, lo);
            tmem_wait_st();
            tc_fence_before();
            mbar_arrive(smem_u32(&sm.a1_full));
            // ---- [B] under this tile's MMA1: once MMA3 of the previous tile is done (its smem operands are free) stage a0^T
            //          (B operand of this tile's MMA3; hi/lo die here), then run the previous tile's dWo phase
            if (it > 0) {
                mbar_wait(smem_u32(&sm.d3_full), ph ^ 1);
                tc_fence_after();
            }
#pragma unroll
            for (int i = 0; i < NC; ++i) {
                sm.sH_hi[tidx(c0 + i, r)] = __uint_as_float(hi[i]);
                sm.sH_lo[tidx(c0 + i, r)] = __uint_as_float(lo[i]);
            }
            if (!EXT && it > 0) dwo_phase(t - gridDim.x, ph ^ 1);
            // ---- [D] epiC
            uint32_t dhv[NC];
            if (EXT) {                                         // dh of this (row, feature) straight from the caller's GEMM; the loads
                const float4 *src = reinterpret_cast<const float4 *>(a.dh_ext + ((size_t)row * a.G + g) * HID + c0);   // fly under MMA1
#pragma unroll
                for (int j4 = 0; j4 < NC / 4; ++j4) {
                    const float4 v = row < nrow ? __ldg(src + j4) : make_float4(0.f, 0.f, 0.f, 0.f);
                    dhv[j4 * 4 + 0] = __float_as_uint(v.x); dhv[j4 * 4 + 1] = __float_as_uint(v.y);
                    dhv[j4 * 4 + 2] = __float_as_uint(v.z); dhv[j4 * 4 + 3] = __float_as_uint(v.w);
                }
            }
            mbar_wait(smem_u32(&sm.d1_full), ph);
            tc_fence_after();
            {
                uint32_t d[NC];
                IO::ld(lane_base + (ph ? colD1b : colD1) + c0, d);
                if (!EXT) IO::ld(lane_base + colDH + c0, dhv);
                tmem_wait_ld();
                float dz[NC];
#pragma unroll
                for (int j4 = 0; j4 < NC / 4; ++j4) {
                    const float4 b = *reinterpret_cast<const float4 *>(sm.b2 + c0 + j4 * 4);
                    const float bb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int jj = j4 * 4 + e;
                        const float act = fmaxf(__uint_as_float(d[jj]) + bb[e], 0.f);
                        float m = act > 0.f ? 1.f : 0.f;
                        if (DROP) m *= gnan_dropout_mul(a.seed, tc_drop_key(a, 1, g, row, c0 + jj), a.drop_thresh, a.drop_scale);
                        dz[jj] = __uint_as_float(dhv[jj]) * m;
                        split_tf32(dz[jj], hi[jj], lo[jj]);
                        if (EXT) d[jj] = __float_as_uint(act * m);           // a1 (after dropout) for the caller's dWo GEMM
                    }
                }
                if (EXT && row < nrow) {
                    float4 *dst = reinterpret_cast<float4 *>(a.a1_ext + ((size_t)row * a.G + g) * HID + c0);
#pragma unroll
                    for (int j4 = 0; j4 < NC / 4; ++j4)
                        dst[j4] = make_float4(__uint_as_float(d[j4 * 4 + 0]), __uint_as_float(d[j4 * 4 + 1]),
                                              __uint_as_float(d[j4 * 4 + 2]), __uint_as_float(d[j4 * 4 + 3]));
                }
                IO::st(lane_base + colA_hi + c0, hi);
                if (!a.single_pass) IO::st(lane_base + colA_lo + c0, lo);
                tmem_wait_st();
                tc_fence_before();
                mbar_arrive(smem_u32(&sm.a2_full));                  // MMA2 may start
#pragma unroll
                for (int jj = 0; jj < NC; ++jj) {                     // transposed staging for MMA3 (off the MMA2 critical path)
                    sm.sZ[tidx(c0 + jj, r)] = __uint_as_float(hi[jj]);
                    sm.sZ[tidx(64 + c0 + jj, r)] = __uint_as_float(lo[jj]);
                }
                fence_async_smem();
                mbar_arrive(smem_u32(&sm.a3_full));                  // MMA3 may start (after MMA2 in issue order)
                p_b2 += warp_colsum<NC>(dz, lane);
            }
            // ---- [E] epiF
            mbar_wait(smem_u32(&sm.d2_full), ph);
            tc_fence_after();
            {
                uint32_t d[NC];
                IO::ld(lane_base + colD2 + c0, d);
                tmem_wait_ld();
                float z0[NC], z1[NC];
#pragma unroll
                for (int i4 = 0; i4 < NC / 4; ++i4) {
                    const float4 w = *reinterpret_cast<const float4 *>(sm.w1 + c0 + i4 * 4);
                    const float4 b = *reinterpret_cast<const float4 *>(sm.b1 + c0 + i4 * 4);
                    const float pre[4] = {fmaf(x, w.x, b.x), fmaf(x, w.y, b.y), fmaf(x, w.z, b.z), fmaf(x, w.w, b.w)};
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int ii = i4 * 4 + e;
                        float m = pre[e] > 0.f ? 1.f : 0.f;
                        if (DROP) m *= gnan_dropout_mul(a.seed, tc_drop_key(a, 0, g, row, c0 + ii), a.drop_thresh, a.drop_scale);
                        z0[ii] = __uint_as_float(d[ii]) * m;
                        z1[ii] = z0[ii] * x;
                    }
                }
                p_b1 += warp_colsum<NC>(z0, lane);
                p_w1 += warp_colsum<NC>(z1, lane);
            }
        }
        // the last tile's dWo phase
        if (it > 0) {
            const int64_t tl = (int64_t)blockIdx.x + (int64_t)(it - 1) * gridDim.x;
            mbar_wait(smem_u32(&sm.d3_full), (it - 1) & 1);
            tc_fence_after();
            if (!EXT) dwo_phase(tl, (it - 1) & 1);
        }
        // ---- write this CTA's partial gradients (everything but dW2)
        const size_t off = (size_t)(blockIdx.x + a.chunk_off) * gp.chunk_stride;
        float *red = &sm.red[0][0];                        // red[warp][0..NC) and [NC..2NC)
        const int lc = lane & (NC - 1);
        // unit u = part*NC + lc lives in the four warps part*4 + q, q = 0..3
        named_bar_sync(1, BWD_ROW_THREADS);
        if (lane < NC) red[warp * 2 * NC + lc] = p_b2;
        named_bar_sync(1, BWD_ROW_THREADS);
        if (tid < HID && gp.bh) {
            float s = 0.f;
            for (int w = 0; w < 4; ++w) s += red[((tid / NC) * 4 + w) * 2 * NC + (tid % NC)];
            gp.bh[off + (size_t)g * HID + tid] = s;
        }
        named_bar_sync(1, BWD_ROW_THREADS);
        if (lane < NC) { red[warp * 2 * NC + lc] = p_b1; red[warp * 2 * NC + NC + lc] = p_w1; }
        named_bar_sync(1, BWD_ROW_THREADS);
        if (tid < HID) {
            float s0 = 0.f, s1 = 0.f;
            for (int w = 0; w < 4; ++w) {
                s0 += red[((tid / NC) * 4 + w) * 2 * NC + (tid % NC)];
                s1 += red[((tid / NC) * 4 + w) * 2 * NC + NC + (tid % NC)];
            }
            if (gp.b1) gp.b1[off + (size_t)g * HID + tid] = s0;
            if (gp.w1) gp.w1[off + (size_t)g * HID + tid] = s1;
        }
        named_bar_sync(1, BWD_ROW_THREADS);
        // dWo: thread holds row group (tid>>6) of unit (tid&63) -> sum the row groups
        constexpr int NRG = BWD_ROW_THREADS / 64;
        float *scr = sm.sZ;
#pragma unroll
        for (int c = 0; c < CT; ++c) scr[(c * NRG + (tid >> 6)) * HID + (tid & 63)] = acc_wo[c];
        named_bar_sync(1, BWD_ROW_THREADS);
        if (gp.wo)
            for (int idx = tid; idx < a.C * HID; idx += BWD_ROW_THREADS) {
                const int c = idx >> 6, j = idx & 63;
                float s = 0.f;
                for (int k = 0; k < NRG; ++k) s += scr[(c * NRG + k) * HID + j];
                gp.wo[off + ((size_t)g * a.Ctot + a.c_off) * HID + idx] = s;
            }
        named_bar_sync(1, BWD_ROW_THREADS);
        // ---- dW2 = D3[lane j] + D3[lane 64 + j]  (hi and lo halves of the stacked A operand); all MMAs are complete (d3_full)
        if (part == 0) {           // warps 0-3 cover all 128 lanes
#pragma unroll
            for (int hc = 0; hc < 2; ++hc) {       // two passes of 32 columns keep the register footprint small
                uint32_t d[32];
                tmem_ld32(lane_base + colD3 + hc * 32, d);
                tmem_wait_ld();
                if (it == 0) {                     // entries mode: a CTA beyond its group's tiles issued no MMA (D3 is undefined)
#pragma unroll
                    for (int i = 0; i < 32; ++i) d[i] = 0u;
                }
                if (r >= 64) {
#pragma unroll
                    for (int i = 0; i < 32; i += 4)
                        *reinterpret_cast<float4 *>(scr + (r - 64) * 36 + i) =
                            make_float4(__uint_as_float(d[i]), __uint_as_float(d[i + 1]), __uint_as_float(d[i + 2]), __uint_as_float(d[i + 3]));
                }
                named_bar_sync(2, 128);
                if (r < 64 && gp.wh) {
                    float *dst = gp.wh + off + ((size_t)g * HID + r) * HID + hc * 32;
#pragma unroll
                    for (int i = 0; i < 32; i += 4) {
                        const float4 o = *reinterpret_cast<const float4 *>(scr + r * 36 + i);
                        *reinterpret_cast<float4 *>(dst + i) = make_float4(__uint_as_float(d[i]) + o.x, __uint_as_float(d[i + 1]) + o.y,
                                                                           __uint_as_float(d[i + 2]) + o.z, __uint_as_float(d[i + 3]) + o.w);
                    }
                }
                named_bar_sync(2, 128);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == BWD_ROW_WARPS) tmem_dealloc(tmem, 512);
}

// d bo[g][c] = sum_r dS[r][c] for every group g (the output bias gradient does not depend on the group)
__global__ void dbo_colsum_kernel(const float *__restrict__ dS, int64_t R, int C, int G, float *__restrict__ dbo)
{
    __shared__ float red[256];
    const int c = blockIdx.x;
    float s = 0.f;
    for (int64_t r = threadIdx.x; r < R; r += blockDim.x) s += dS[r * C + c];
    red[threadIdx.x] = s;
    __syncthreads();
    for (int k = 128; k > 0; k >>= 1) {
        if ((int)threadIdx.x < k) red[threadIdx.x] += red[threadIdx.x + k];
        __syncthreads();
    }
    for (int g = threadIdx.x; g < G; g += blockDim.x) dbo[(size_t)g * C + c] = red[0];
}

// entries mode: d bo[g][c] = sum over the entries of group g; one warp per (g, c), fixed order (lane-strided partial sums, then
// a butterfly): deterministic. Groups are short at bag-of-words shapes (35 entries) and long for one-hot ones (9 k).
__global__ void dbo_entries_kernel(const float *__restrict__ dY, const int64_t *__restrict__ grp_ptr, int G, int C, float *__restrict__ dbo)
{
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= (int64_t)G * C) return;
    const int g = (int)(w / C), c = (int)(w % C);
    float s0 = 0.f, s1 = 0.f;
    const int64_t e1 = grp_ptr[g + 1];
    int64_t e = grp_ptr[g] + lane;
    for (; e + 32 < e1; e += 64) { s0 += dY[e * C + c]; s1 += dY[(e + 32) * C + c]; }
    if (e < e1) s0 += dY[e * C + c];
    float s = s0 + s1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) dbo[w] = s;
}

struct TcFwdPlan { int KC, nchunk; int64_t ntile; };

TcFwdPlan plan_tc_fwd(int64_t R, const gnan_mlp_params *p)
{
    TcFwdPlan pl;
    pl.ntile = ceil_div64(R, FWD_GROUPS * ROWS);
    const int target = 2 * gnan_sm_count();                    // ~2 waves of one CTA per SM
    int nchunk = (int)std::max<int64_t>(1, std::min<int64_t>(p->G, ceil_div64(target, pl.ntile)));
    pl.KC = (int)ceil_div64(p->G, nchunk);
    if (pl.KC < 8) pl.KC = std::min(8, (int)p->G);             // amortise the CTA prologue (TMEM allocation, barriers)
    pl.nchunk = (int)ceil_div64(p->G, pl.KC);
    return pl;
}

TcArgs make_tc_args(const float *u, int64_t R, int64_t ldu, const gnan_mlp_params *p, float dropout_p, uint64_t seed, int precision)
{
    TcArgs a;
    a.u = u; a.R = R; a.ldu = ldu; a.G = p->G; a.C = p->C;
    a.w1 = p->w1; a.b1 = p->b1; a.wh = p->wh; a.bh = p->bh; a.wo = p->wo; a.bo = p->bo;
    a.drop_thresh = dropout_p > 0.f ? gnan_dropout_thresh(dropout_p) : 0u;
    a.drop_scale = dropout_p > 0.f ? 1.f / (1.f - dropout_p) : 1.f;
    a.seed = seed;
    a.seed_dev = nullptr;
    a.single_pass = precision == GNAN_PREC_TF32;
    a.grp_ptr = nullptr;
    a.Ctot = p->C; a.c_off = 0; a.chunk_off = 0;
    a.dh_ext = nullptr; a.a1_ext = nullptr;
    return a;
}

template <int CP>
int launch_tc_fwd_cp(const TcArgs &a, const TcFwdPlan &pl, float *Spart, cudaStream_t st)
{
    const size_t smem = sizeof(FwdSmem<CP>) + 1024;
    dim3 grid((unsigned)pl.ntile, (unsigned)pl.nchunk);
    if (a.drop_thresh) {
        GNAN_CUDA(cudaFuncSetAttribute(mlp_tc_fwd_kernel<true, CP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        mlp_tc_fwd_kernel<true, CP><<<grid, FWD_THREADS, smem, st>>>(a, pl.KC, Spart);
    } else {
        GNAN_CUDA(cudaFuncSetAttribute(mlp_tc_fwd_kernel<false, CP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        mlp_tc_fwd_kernel<false, CP><<<grid, FWD_THREADS, smem, st>>>(a, pl.KC, Spart);
    }
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}

int launch_tc_fwd(const TcArgs &a, const TcFwdPlan &pl, float *Spart, cudaStream_t st)
{
    if (a.C <= 8) return launch_tc_fwd_cp<8>(a, pl, Spart, st);
    if (a.C <= 16) return launch_tc_fwd_cp<16>(a, pl, Spart, st);
    if (a.C <= 32) return launch_tc_fwd_cp<32>(a, pl, Spart, st);
    if (a.C <= 48) return launch_tc_fwd_cp<48>(a, pl, Spart, st);
    return launch_tc_fwd_cp<64>(a, pl, Spart, st);
}

}  // namespace

int gnan_mlp_tc_supported(const gnan_mlp_params *p, int precision)
{
    return (precision == GNAN_PREC_TF32X3 || precision == GNAN_PREC_TF32) && p->H == HID && p->n_layers == 3 && p->C <= CF_MAX;
}

int gnan_mlp_tc_bwd_supported(const gnan_mlp_params *p, int precision) { return gnan_mlp_tc_supported(p, precision); }

// backward passes over 8-channel slices
static inline int tc_bwd_passes(const gnan_mlp_params *p) { return (p->C + CT_MAX - 1) / CT_MAX; }

namespace {
inline size_t pad4(size_t n) { return (n + 3) / 4 * 4; }
size_t tc_grad_floats(const gnan_mlp_params *p)
{
    const size_t G = p->G, C = p->C;
    return 2 * pad4(G * HID) + pad4(G * HID * HID) + pad4(G * HID) + pad4(G * C * HID) + pad4(G * C);
}
struct TcBwdPlan { int nchunk; int64_t ntile; };
TcBwdPlan plan_tc_bwd(int64_t R, const gnan_mlp_params *p)
{
    TcBwdPlan pl;
    pl.ntile = ceil_div64(R, ROWS);
    int nchunk = (int)ceil_div64(2 * gnan_sm_count(), p->G);
    // every CTA stages the feature's weights and writes a partial gradient set: give it at least 4 tiles, which also keeps
    // the partial-gradient reduction short (G = 1, the rho table, used to produce 254 chunks of 4.6 k floats)
    nchunk = (int)std::min<int64_t>(nchunk, std::max<int64_t>(1, pl.ntile / 4));
    pl.nchunk = std::max(nchunk, 1);
    return pl;
}
int launch_tc_bwd_ext(const TcArgs &a, const TcBwdPlan &pl, const float *dS, const TcGradPtrs &gp, cudaStream_t st)
{
    const size_t smem = sizeof(BwdSmem) + 1024;
    dim3 grid((unsigned)pl.nchunk, (unsigned)a.G);
    if (a.drop_thresh) {
        GNAN_CUDA(cudaFuncSetAttribute(mlp_tc_bwd_kernel<1, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        mlp_tc_bwd_kernel<1, true, true><<<grid, BWD_THREADS, smem, st>>>(a, dS, gp, pl.ntile);
    } else {
        GNAN_CUDA(cudaFuncSetAttribute(mlp_tc_bwd_kernel<1, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        mlp_tc_bwd_kernel<1, false, true><<<grid, BWD_THREADS, smem, st>>>(a, dS, gp, pl.ntile);
    }
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}

template <int CT>
int launch_tc_bwd(const TcArgs &a, const TcBwdPlan &pl, const float *dS, const TcGradPtrs &gp, cudaStream_t st)
{
    const size_t smem = sizeof(BwdSmem) + 1024;
    dim3 grid((unsigned)pl.nchunk, (unsigned)a.G);
    if (a.drop_thresh) {
        GNAN_CUDA(cudaFuncSetAttribute(mlp_tc_bwd_kernel<CT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        mlp_tc_bwd_kernel<CT, true><<<grid, BWD_THREADS, smem, st>>>(a, dS, gp, pl.ntile);
    } else {
        GNAN_CUDA(cudaFuncSetAttribute(mlp_tc_bwd_kernel<CT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        mlp_tc_bwd_kernel<CT, false><<<grid, BWD_THREADS, smem, st>>>(a, dS, gp, pl.ntile);
    }
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}
}  // namespace

size_t gnan_mlp_tc_workspace_bytes(int64_t R, const gnan_mlp_params *p, int backward, int precision)
{
    (void)precision;
    if (backward) {
        const TcBwdPlan pl = plan_tc_bwd(R, p);
        const int slots = pl.nchunk * tc_bwd_passes(p);
        return slots > 1 ? sizeof(float) * (size_t)slots * tc_grad_floats(p) : 0;
    }
    const TcFwdPlan pl = plan_tc_fwd(R, p);
    return pl.nchunk > 1 ? sizeof(float) * (size_t)pl.nchunk * R * p->C : 0;
}

int gnan_mlp_tc_fwd(const float *u, int64_t R, int64_t ldu, const gnan_mlp_params *p, float dropout_p, uint64_t seed,
                    int precision, float *S, void *ws, size_t ws_bytes, cudaStream_t st, const uint64_t *seed_dev)
{
    const TcFwdPlan pl = plan_tc_fwd(R, p);
    float *Spart = S;
    if (pl.nchunk > 1) {
        const size_t need = sizeof(float) * (size_t)pl.nchunk * R * p->C;
        if (!ws || ws_bytes < need) {
            gnan_set_error("mlp_fwd(tc): workspace %zu < %zu bytes", ws_bytes, need);
            return GNAN_ERR_WORKSPACE;
        }
        Spart = (float *)ws;
    }
    TcArgs a = make_tc_args(u, R, ldu, p, dropout_p, seed, precision);
    a.seed_dev = seed_dev;
    int rc = launch_tc_fwd(a, pl, Spart, st);
    if (rc) return rc;
    if (pl.nchunk > 1) return gnan_reduce_chunks(Spart, pl.nchunk, (size_t)R * p->C, (size_t)R * p->C, S, st);
    return GNAN_OK;
}

// entries-mode forward on tcgen05 (H = 64, 3 layers, C <= 8): Y[e,:] = f_g(val[e]); items [n_items][2] = (group, tile)
int gnan_mlp_tc_entries_fwd_supported(const gnan_mlp_params *p, int precision)
{
    return gnan_mlp_tc_supported(p, precision) && p->C <= CT_MAX;
}

int gnan_mlp_tc_entries_fwd(const float *val, const int64_t *grp_ptr, int64_t E, const int32_t *items, int64_t n_items,
                            const gnan_mlp_params *p, int precision, float *Y, cudaStream_t st)
{
    TcArgs a = make_tc_args(val, E, 1, p, 0.f, 0, precision);
    a.grp_ptr = grp_ptr;
    const size_t smem = sizeof(EntSmem) + 1024;
    GNAN_CUDA(cudaFuncSetAttribute(mlp_tc_entries_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int grid = (int)std::min<int64_t>(gnan_sm_count(), ceil_div64(n_items, FWD_GROUPS));
    mlp_tc_entries_fwd_kernel<<<grid, ENT_THREADS, smem, st>>>(a, items, n_items, Y);
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}

// grp_ptr != NULL: entries mode, u = val[E], R = the largest group (sizes the row chunks), dS = dY[E,C]
int gnan_mlp_tc_bwd_ex(const float *u, int64_t R, int64_t ldu, const gnan_mlp_params *p, float dropout_p, uint64_t seed,
                       int precision, const float *dS, const gnan_mlp_grads *grads, void *ws, size_t ws_bytes, cudaStream_t st,
                       const int64_t *grp_ptr, const uint64_t *seed_dev, const float *dh_ext, float *a1_ext)
{
    const TcBwdPlan pl = plan_tc_bwd(R, p);
    const size_t G = p->G, C = p->C, ntot = tc_grad_floats(p);
    const bool ext = dh_ext != nullptr && a1_ext != nullptr && grp_ptr == nullptr;      // output layer outside: one pass for any C
    const int npass = ext ? 1 : tc_bwd_passes(p), slots = pl.nchunk * npass;
    TcGradPtrs gp;
    if (slots > 1) {
        const size_t need = sizeof(float) * (size_t)slots * ntot;
        if (!ws || ws_bytes < need) {
            gnan_set_error("mlp_bwd(tc): workspace %zu < %zu bytes", ws_bytes, need);
            return GNAN_ERR_WORKSPACE;
        }
        float *w = (float *)ws;
        gp.w1 = w; w += pad4(G * HID);
        gp.b1 = w; w += pad4(G * HID);
        gp.wh = w; w += pad4(G * HID * HID);
        gp.bh = w; w += pad4(G * HID);
        gp.wo = w; w += pad4(G * C * HID);
        gp.bo = w;
        gp.chunk_stride = ntot;
    } else {
        gp.w1 = grads->w1; gp.b1 = grads->b1; gp.wh = grads->wh; gp.bh = grads->bh; gp.wo = grads->wo; gp.bo = grads->bo;
        gp.chunk_stride = 0;
    }
    TcArgs a = make_tc_args(u, R, ldu, p, dropout_p, seed, precision);
    a.grp_ptr = grp_ptr;
    a.seed_dev = seed_dev;
    int rc = GNAN_OK;
    if (npass > 1)     // a pass writes only its own channel slice of dWo: the other slots' slices must read as zero in the reduction
        GNAN_CUDA(cudaMemsetAsync(ws, 0, sizeof(float) * (size_t)slots * ntot, st));
    if (ext) {
        a.dh_ext = dh_ext; a.a1_ext = a1_ext;
        gp.wo = nullptr;                                        // dWo = dS^T a1 is the caller's GEMM
        rc = launch_tc_bwd_ext(a, pl, dS, gp, st);
    }
    for (int ps = 0; ps < npass && !rc && !ext; ++ps) {
        a.c_off = ps * CT_MAX;
        a.C = std::min<int>(CT_MAX, (int)C - a.c_off);
        a.chunk_off = ps * pl.nchunk;
        if (a.C == 1) rc = launch_tc_bwd<1>(a, pl, dS, gp, st);
        else if (a.C == 2) rc = launch_tc_bwd<2>(a, pl, dS, gp, st);
        else if (a.C <= 4) rc = launch_tc_bwd<4>(a, pl, dS, gp, st);
        else rc = launch_tc_bwd<8>(a, pl, dS, gp, st);
    }
    if (rc) return rc;
    if (slots > 1) {
        GnanReduceSegs sg{};                                    // the five gradient arrays in one launch
        sg.add(gp.w1, grads->w1, G * HID); sg.add(gp.b1, grads->b1, G * HID); sg.add(gp.wh, grads->wh, G * HID * HID);
        sg.add(gp.bh, grads->bh, G * HID);
        if (!ext) sg.add(gp.wo, grads->wo, G * C * HID);
        rc = gnan_reduce_chunks_multi(sg, slots, ntot, st);
        if (rc) return rc;
    }
    if (grads->bo) {
        if (grp_ptr) dbo_entries_kernel<<<(unsigned)ceil_div64((int64_t)G * C * 32, 256), 256, 0, st>>>(dS, grp_ptr, (int)G, (int)C, grads->bo);
        else dbo_colsum_kernel<<<(unsigned)C, 256, 0, st>>>(dS, R, (int)C, (int)G, grads->bo);
        GNAN_LAUNCH_OK();
    }
    return GNAN_OK;
}
