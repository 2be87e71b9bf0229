// Tensor-core aggregation over the uint8 hop matrix: one pass over the hop bytes for ALL channels.
//
// Reference lines replaced: GNAN.py:64-73 (rho on N*N pairs, permute, matmul(m_dist_perm, fx_perm), sum), GNAN.py:159-170,
// models.py:366-375; backward = autograd through the same.
//
// Distance-class form.  With b(h) the bin of a hop byte, the reference's [C,N,N] x [C,N,K] contraction is
//     Bsum[i,d,c] = sum_j 1[b(hop[i,j]) = d] * S[j,c]            (a GEMM with a 0/1 operand)
//     out[i,c]    = sum_d T[ti,d,c'] * rscale[i,d] * Bsum[i,d,c]
// Bsum is also everything the backward needs for dT.  The 0/1 operand is generated on the fly and never exists in memory:
//   * the hop tile [rows x 128 columns] lands in shared memory by TMA (cp.async.bulk.tensor.2d, uint8 tensor map);
//   * a generator thread owns one TMEM lane = one (row, bin) pair. The hop bytes of its row are packed to 4-bit selectors
//     once per tile (cooperatively), and ONE `prmt` with a per-thread 8-byte lookup table (0x01 at byte bin%8) turns four
//     selectors into four int8 one-hot values (selector bit 3 = "other half of the bins" -> 0 through prmt's sign-replicate
//     mode). The values go straight into tensor memory with tcgen05.st: the A operand never touches shared memory;
//   * S is quantised per channel to ndig signed 8-bit digits of a common power-of-two scale (exact integer arithmetic:
//     S*2^sh rounded once, abs. error <= 2^-31 (4 digits) or 2^-23 (3 digits) of the column maximum); the digit matrix is the
//     B operand, pre-laid-out in the UMMA K-major core-matrix order by a small pre-pass so that a stage is one bulk copy;
//   * tcgen05.mma kind::i8 accumulates int32 in TMEM over the whole row sweep: the bin sums are EXACT sums of the quantised
//     values, independent of summation order (deterministic), and are rounded to fp32 once in the epilogue.
// Cost per hop byte: ~0.5 ALU instructions per (pair, bin) + NP*NB/256 tensor cycles per 32 bytes, independent of C up to
// NP = 16*ceil(C/4|5) accumulator columns.
//
// Backward dS[j,c] = sum_{i,d} 1[b(hop[i,j]) = d] * TG[i,d,c],  TG = T*rscale*g: the same machinery transposed (a TMEM lane
// = a hop COLUMN j, the contraction index is (row, bin)); rows whose g is entirely zero are skipped (exact): with a
// train-mask loss that is almost all of them.
#include <cuda.h>

#include <algorithm>
#include <cmath>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace {

constexpr int TCOLS = 128;        // hop columns per pipeline stage (TMA box inner extent, bytes)
constexpr int MAX_STAGES = 16;

// ---- PTX: TMA + the i8 MMA -------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, int c0, int c1, uint32_t bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 :: "r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(bar) : "memory");
}
__device__ __forceinline__ void bulk_load_1d(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap *map)
{
    asm volatile("prefetch.tensormap [%0];" :: "l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
// generic-mode prmt: selector nibble bit 3 replicates the msb of the selected byte (0 for our 0x00/0x01 table)
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel)
{
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}
// instruction descriptor, kind::i8: signed 8-bit A and B (K-major), int32 accumulate
__host__ __device__ constexpr uint32_t umma_idesc_i8(int M, int N)
{
    return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_i8_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accum)
{
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, p;\n\t}\n"
                 :: "r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accum) : "memory");
}

// B operand of one stage: NP rows (accumulator columns) x 128 K-bytes, UMMA K-major no-swizzle core matrices
// (8 rows x 16 bytes = 128 contiguous bytes); K-adjacent core matrices 128 B apart (LBO), 8-row groups 1024 B apart (SBO)
constexpr uint32_t DG_LBO = 128, DG_SBO = 1024, DG_KSTEP = 256;
__host__ __device__ inline size_t digit_offset(int n, int k) { return (size_t)(n >> 3) * 1024 + (k >> 4) * 128 + (n & 7) * 16 + (k & 15); }

// digit layout along the accumulator columns: a 16-column chunk holds CPC channels x ndig digits (never straddles a chunk)
struct DigitPlan { int ndig, cpc, NP; };
inline DigitPlan digit_plan(int C)
{
    const int c4 = (C + 3) / 4, c5 = (C + 4) / 5;
    DigitPlan p;
    if (c4 == c5) { p.ndig = 4; p.cpc = 4; p.NP = 16 * c4; }
    else { p.ndig = 3; p.cpc = 5; p.NP = 16 * c5; }
    return p;
}

// ---- pre-pass: per-channel scale and the digit matrix -------------------------------------------------------------------
__global__ void colmax_kernel(const float *__restrict__ S, int64_t n_rows, int C, uint32_t *__restrict__ colmax)
{
    // |x| as uint32 orders like the float for non-negative values; one atomicMax per warp and channel
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int c = 0; c < C; ++c) {
        uint32_t m = 0;
        for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n_rows; j += stride)
            m = max(m, __float_as_uint(fabsf(S[j * C + c])));
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, s));
        if ((threadIdx.x & 31) == 0 && m) atomicMax(colmax + c, m);
    }
}

// shift sh such that |x * 2^sh| <= 2^(8*ndig-2) for every |x| <= colmax
__device__ __forceinline__ int digit_shift(uint32_t colmax_bits, int ndig)
{
    if (colmax_bits == 0) return 0;
    const int e = (int)((colmax_bits >> 23) & 0xff) - 127 + 1;       // colmax < 2^e  (subnormal colmax: e = -126, harmless)
    return 8 * ndig - 2 - e;
}

// one thread per (column block, accumulator column n, k): Sdig[blk][digit_offset(n,k)]; row_map (optional) gathers rows
__global__ void digits_kernel(const float *__restrict__ X, int64_t n_rows, int C, int ld_x, const int32_t *__restrict__ row_map,
                              const uint32_t *__restrict__ colmax, int ndig, int cpc, int NP, int8_t *__restrict__ dig,
                              int32_t *__restrict__ colsh)
{
    const int blk = blockIdx.x;
    if (blk == 0 && threadIdx.x < C) colsh[threadIdx.x] = digit_shift(colmax[threadIdx.x], ndig);
    for (int t = threadIdx.x; t < NP * TCOLS; t += blockDim.x) {
        const int n = t / TCOLS, k = t % TCOLS;
        const int64_t j = (int64_t)blk * TCOLS + k;
        const int chunk = n >> 4, w = n & 15, cc = w / ndig, kd = w % ndig;
        const int c = chunk * cpc + cc;
        int8_t v = 0;
        if (j < n_rows && cc < cpc && c < C) {
            const int64_t src = row_map ? row_map[j] : j;
            const float x = X[src * ld_x + c];
            const int sh = digit_shift(colmax[c], ndig);
            long long q = __double2ll_rn(ldexp((double)x, sh));
            for (int s = 0; s < kd; ++s) {                      // balanced base-256 digits in [-128, 127]
                const long long b = ((q + 128) & 255) - 128;
                q = (q - b) >> 8;
            }
            v = (int8_t)(((q + 128) & 255) - 128);
            if (kd == ndig - 1) v = (int8_t)q;                   // top digit carries the rest (|q| <= 65 by construction)
        }
        dig[(size_t)blk * NP * TCOLS + digit_offset(n, k)] = v;
    }
}

// ---- forward -------------------------------------------------------------------------------------------------------------
struct AggTcArgs {
    int64_t R, N;
    int nbins, C, Cr, per_row, ndig, cpc, NP, nblk, stages;
    const float *T, *rscale;
    const int32_t *colsh;
    const int8_t *dig;
    float *out, *Bsum;
};

// 8 hop bytes -> the two 4-selector words of one stream (selector k of a word in nibble k, upper 16 bits zero: prmt reads only
// the low 16 bits of its selector operand); NB = bins per row slot
template <int NBX>
__device__ __forceinline__ uint2 pack8(uint2 w, int stream)
{
    constexpr int NB = NBX <= 8 ? 8 : (NBX <= 16 ? 16 : 32);      // selector width: 9..16 lanes per row use the 4-bit selectors
    uint32_t a = w.x, b = w.y;
    if (NB == 32) {
        const uint32_t q = 0x01010101u * (uint32_t)stream;
        const uint32_t a5 = a & 0x1f1f1f1fu, b5 = b & 0x1f1f1f1fu;
        uint32_t xa = ((a5 >> 3) & 0x03030303u) ^ q, xb = ((b5 >> 3) & 0x03030303u) ^ q;
        xa = (xa | (xa >> 1)) & 0x01010101u;
        xb = (xb | (xb >> 1)) & 0x01010101u;
        a = (a5 & 0x07070707u) | (xa << 3);
        b = (b5 & 0x07070707u) | (xb << 3);
    }
    // byte k of a/b holds selector k in its low nibble (NB <= 16: hop & 15 / & 7; 255 = unreachable -> the last slot):
    // merge neighbours into bytes 0 and 2 (low nibble = even selector, high nibble = odd selector), then gather those bytes
    constexpr uint32_t LO = NB == 8 ? 0x07070707u : 0x0f0f0f0fu, HI = NB == 8 ? 0x70707070u : 0xf0f0f0f0u;
    a = (a & LO) | ((a >> 4) & HI);
    b = (b & LO) | ((b >> 4) & HI);
    uint32_t lo = prmt(a, 0u, 0x4420u), hi = prmt(b, 0u, 0x4420u);
    if (NB == 16 && stream) { lo ^= 0x8888u; hi ^= 0x8888u; }
    return make_uint2(lo, hi);
}

constexpr int NBUF = 3;            // A-operand buffers per generator group in tensor memory

// NB = TMEM lanes per hop row (bin slots). 8 / 16 / 32 tile the 128 lanes exactly; 10 / 12 / 14 (levels + unreachable of a
// 9..15-bin table) leave 128 % NB lanes idle but put 128 / NB instead of 8 rows into every MMA: with many channels the pass
// is bound by the int8 tensor pipe, whose work per hop byte is NB x digit columns.
template <int NB, int NGR>
struct TcCfg {
    static constexpr int RG = 128 / NB;             // hop rows per generator group (one MMA: M = 128 >= RG rows x NB bins)
    static constexpr int ROWS = RG * NGR;           // hop rows per CTA
    static constexpr int NBP = NB <= 8 ? 8 : (NB <= 16 ? 16 : 32);   // selector space (power of two)
    static constexpr int NSTREAM = NBP / 8;         // selector streams (one per group of 8 bins)
    static constexpr int HOPB = ROWS * TCOLS;       // hop bytes per stage
    static constexpr int RW = (32 % NB == 0) ? 32 / NB : 4;   // hop rows whose lanes fall into one generator warp (at most)
    static constexpr int NIB_WARP = NSTREAM * RW * 32;        // words per warp and buffer: [stream][row of the warp][32 selector words]
    static constexpr int NIB_BUF = 4 * NIB_WARP;              // per group: the four generator warps keep PRIVATE copies of their rows
    static constexpr int NIB_WORDS = 2 * NIB_BUF;             // double-buffered
    static constexpr int ACC0 = NGR * NBUF * 32;    // TMEM: A buffers [g][buf] 32 columns each, then the accumulators
    static constexpr int THREADS = (NGR * 5 + 1) * 32;        // 4 generator warps + 1 MMA-issuer warp per group, 1 TMA producer warp
};

struct PipeBars {
    uint64_t *full, *empty, *a_full, *a_empty, *acc_full;
    uint32_t *tmem_slot;
};

template <int NGR>
__device__ __forceinline__ PipeBars carve_bars(void *base)
{
    PipeBars p;
    p.full = reinterpret_cast<uint64_t *>(base);
    p.empty = p.full + MAX_STAGES;
    p.a_full = p.empty + MAX_STAGES;            // [NGR][NBUF]
    p.a_empty = p.a_full + NGR * NBUF;          // [NGR][NBUF]
    p.acc_full = p.a_empty + NGR * NBUF;        // [NGR]
    p.tmem_slot = reinterpret_cast<uint32_t *>(p.acc_full + NGR);
    return p;
}
constexpr size_t pipe_bar_bytes(int ngr) { return sizeof(uint64_t) * (2 * MAX_STAGES + 2 * ngr * NBUF + ngr) + 16; }

template <int NGR>
__device__ __forceinline__ uint32_t pipe_setup(const PipeBars &p, int stages)
{
    const int tid = threadIdx.x, warp = tid >> 5;
    if (warp == 0) tmem_alloc(smem_u32(p.tmem_slot), 512);
    if (tid == 32) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(smem_u32(&p.full[s]), 1);
            mbar_init(smem_u32(&p.empty[s]), NGR);       // one tcgen05.commit per group
        }
        for (int g = 0; g < NGR * NBUF; ++g) {
            mbar_init(smem_u32(&p.a_full[g]), 128);
            mbar_init(smem_u32(&p.a_empty[g]), 1);
        }
        for (int g = 0; g < NGR; ++g) mbar_init(smem_u32(&p.acc_full[g]), 1);
        mbar_init_fence();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    return *p.tmem_slot;
}

// the MMA issuer of group g: stage s -> 4 x (M128, N = NP, K32) on A buffer s % NBUF and the stage's B tile
template <int NGR>
__device__ __forceinline__ void issuer_loop(const PipeBars &p, uint32_t tmem, int g, int lane, int nst, int stages, int NP, int acc0,
                                            const uint8_t *b_s, int BB)
{
    const uint32_t idesc = umma_idesc_i8(128, NP);
    int st = 0, buf = 0;
    uint32_t fph = 0, aph = 0;
    for (int s = 0; s < nst; ++s) {
        mbar_wait(smem_u32(&p.a_full[g * NBUF + buf]), aph);
        mbar_wait(smem_u32(&p.full[st]), fph);           // complete long ago (the generators waited on it): orders the B tile for this thread
        tc_fence_after();
        if (lane == 0) {
            const uint32_t bb = smem_u32(b_s + (size_t)st * BB);
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
                umma_i8_ts(tmem + (uint32_t)(acc0 + g * NP), tmem + (uint32_t)((g * NBUF + buf) * 32 + ks * 8),
                           umma_desc_kmajor(bb + ks * DG_KSTEP, DG_LBO, DG_SBO), idesc, (s > 0 || ks > 0) ? 1u : 0u);
            umma_commit(smem_u32(&p.a_empty[g * NBUF + buf]));
            umma_commit(smem_u32(&p.empty[st]));
        }
        __syncwarp();
        if (++st == stages) { st = 0; fph ^= 1u; }
        if (++buf == NBUF) { buf = 0; aph ^= 1u; }
    }
    if (lane == 0 && nst > 0) umma_commit(smem_u32(&p.acc_full[g]));
    __syncwarp();
}

template <int NB, int NGR>
__global__ void __launch_bounds__(TcCfg<NB, NGR>::THREADS, 1)
agg_tc_fwd_kernel(const __grid_constant__ CUtensorMap tmap, AggTcArgs a)
{
    using Cfg = TcCfg<NB, NGR>;
    constexpr int RG = Cfg::RG, NSTREAM = Cfg::NSTREAM, HOPB = Cfg::HOPB;
    extern __shared__ __align__(1024) uint8_t smem[];
    const int BB = a.NP * TCOLS;
    uint8_t *hop_s = smem;
    uint8_t *b_s = hop_s + (size_t)a.stages * HOPB;
    uint32_t *nib_s = reinterpret_cast<uint32_t *>(b_s + (size_t)a.stages * BB);
    const PipeBars pb = carve_bars<NGR>(nib_s + NGR * Cfg::NIB_WORDS);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t row0 = (int64_t)blockIdx.x * Cfg::ROWS;
    const uint32_t tmem = pipe_setup<NGR>(pb, a.stages);

    if (warp < NGR * 4) {
        // ===== generators: thread m of group g owns TMEM lane m = (row r, bin slot) =====
        const int g = warp >> 2, m = tid & 127;
        const int r = m / NB, slot = m % NB;
        const bool lane_used = r < RG;                                // 128 % NB idle lanes store zeros
        // selector value this lane answers to: its slot, except that the last slot is the unreachable bin (hop byte 255, whose
        // low selector bits are all ones)
        const int mv = slot == NB - 1 ? Cfg::NBP - 1 : slot;
        const int strm = mv >> 3;
        const uint32_t lut_lo = (lane_used && (mv & 7) < 4) ? 1u << (8 * (mv & 7)) : 0u;
        const uint32_t lut_hi = (lane_used && (mv & 7) >= 4) ? 1u << (8 * ((mv & 7) - 4)) : 0u;
        const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
        const int wq = warp & 3;
        const int r_lo = (wq * 32) / NB;                              // first hop row with a lane in this warp
        uint32_t *nib_g = nib_s + g * Cfg::NIB_WORDS + wq * Cfg::NIB_WARP;
        int st = 0, buf = 0, prev_buf = 0;
        uint32_t fph = 0, eph = 1;                                   // eph: parity of the a_empty completion that frees `buf` (lap - 1)
        for (int s = 0; s < a.nblk; ++s) {
            mbar_wait(smem_u32(&pb.full[st]), fph);
            // pack: the 32 lanes of a warp are (32 / NB rows) x NB bin slots, so a warp packs exactly the rows its own lanes read:
            // 8 hop bytes -> two 4-selector words per stream, through a warp-private slice of shared memory (__syncwarp only)
            uint32_t *nb = nib_g + (s & 1) * Cfg::NIB_BUF;
            const uint8_t *hs = hop_s + (size_t)st * HOPB + (size_t)g * RG * TCOLS;
            constexpr int CH_W = Cfg::RW * 16;                        // 8-byte chunks of the rows this warp's lanes belong to
#pragma unroll
            for (int cw = lane; cw < CH_W; cw += 32) {
                const int rl = cw >> 4, rr = min(r_lo + rl, RG - 1);  // (rows past the group: a copy of the last one, never read)
                const uint2 w = *reinterpret_cast<const uint2 *>(hs + (rr * 16 + (cw & 15)) * 8);
#pragma unroll
                for (int q = 0; q < NSTREAM; ++q) *reinterpret_cast<uint2 *>(nb + q * (Cfg::RW * 32) + cw * 2) = pack8<NB>(w, q);
            }
            if (s > 0) {                                              // the previous stage's TMEM store has had the pack to land
                tmem_wait_st();
                tc_fence_before();
                mbar_arrive(smem_u32(&pb.a_full[g * NBUF + prev_buf]));
            }
            __syncwarp();
            mbar_wait(smem_u32(&pb.a_empty[g * NBUF + buf]), eph);   // first lap: a fresh barrier passes a wait on parity 1
            tc_fence_after();
            const uint4 *src = reinterpret_cast<const uint4 *>(nb + strm * (Cfg::RW * 32) + (min(r, RG - 1) - r_lo) * 32);
            uint32_t v[32];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const uint4 p = src[q];
                v[4 * q + 0] = prmt(lut_lo, lut_hi, p.x); v[4 * q + 1] = prmt(lut_lo, lut_hi, p.y);
                v[4 * q + 2] = prmt(lut_lo, lut_hi, p.z); v[4 * q + 3] = prmt(lut_lo, lut_hi, p.w);
            }
            tmem_st32(lane_base + (uint32_t)((g * NBUF + buf) * 32), v);
            prev_buf = buf;
            if (++st == a.stages) { st = 0; fph ^= 1u; }
            if (++buf == NBUF) { buf = 0; eph ^= 1u; }
        }
        tmem_wait_st();
        tc_fence_before();
        mbar_arrive(smem_u32(&pb.a_full[g * NBUF + prev_buf]));
        // ===== epilogue: Bsum (exact integer bin sums -> fp32) and out = sum_d T * rscale * Bsum =====
        mbar_wait(smem_u32(&pb.acc_full[g]), 0);
        tc_fence_after();
        const int64_t i = row0 + g * RG + r;
        const bool slot_ok = slot < a.nbins - 1 || slot == NB - 1;
        const int d = slot == NB - 1 ? a.nbins - 1 : slot;
        const bool ok = lane_used && i < a.R && slot_ok;
        constexpr bool POW2 = (NB & (NB - 1)) == 0;
        float *sc = reinterpret_cast<float *>(nib_s + g * Cfg::NIB_WORDS);   // the group's selector buffers are free now: [128][5] scratch
        const float rs = (ok && a.rscale) ? a.rscale[i * a.nbins + d] : 1.f;
        const float *Trow = a.T + ((a.per_row && ok) ? i * a.nbins * a.Cr : 0) + (ok ? d * a.Cr : 0);
        for (int n0 = 0; n0 < a.NP; n0 += 16) {
            uint32_t acc[16];
            tmem_ld16(lane_base + (uint32_t)(Cfg::ACC0 + g * a.NP + n0), acc);
            tmem_wait_ld();
#pragma unroll
            for (int cc = 0; cc < 5; ++cc) {
                const int c = (n0 >> 4) * a.cpc + cc;
                if (cc >= a.cpc || c >= a.C) break;
                long long tot = 0;
                if (a.ndig == 4) {
#pragma unroll
                    for (int k = 3; k >= 0; --k) tot = tot * 256 + (int)acc[(cc * 4 + k) & 15];
                } else {
#pragma unroll
                    for (int k = 2; k >= 0; --k) tot = tot * 256 + (int)acc[(cc * 3 + k) & 15];
                }
                const float bs = (float)ldexp((double)tot, -a.colsh[c]);
                if (ok && a.Bsum) a.Bsum[(i * a.nbins + d) * a.C + c] = bs;
                float o = ok ? Trow[a.Cr == 1 ? 0 : c] * rs * bs : 0.f;
                if (POW2) {
#pragma unroll
                    for (int sft = NB / 2; sft > 0; sft >>= 1) o += __shfl_xor_sync(0xffffffffu, o, sft);
                    if (slot == 0 && i < a.R) a.out[i * a.C + c] = o;
                } else {
                    sc[m * 5 + cc] = o;
                }
            }
            if (!POW2) {                                              // a row's lanes straddle warps: sum them through shared memory
                named_bar_sync(1 + g, 128);
                if (m < RG * 5) {
                    const int rr = m / 5, cc = m % 5;
                    const int c = (n0 >> 4) * a.cpc + cc;
                    const int64_t ii = row0 + g * RG + rr;
                    if (cc < a.cpc && c < a.C && ii < a.R) {
                        float o = 0.f;
#pragma unroll
                        for (int sl = 0; sl < NB; ++sl) o += sc[(rr * NB + sl) * 5 + cc];
                        a.out[ii * a.C + c] = o;
                    }
                }
                named_bar_sync(1 + g, 128);
            }
        }
        tc_fence_before();
    } else if (warp < NGR * 5) {
        issuer_loop<NGR>(pb, tmem, warp - NGR * 4, lane, a.nblk, a.stages, a.NP, Cfg::ACC0, b_s, BB);
    } else {
        // ===== TMA producer =====
        if (lane == 0) {
            prefetch_tmap(&tmap);
            int st = 0;
            uint32_t eph = 1;
            for (int s = 0; s < a.nblk; ++s) {
                mbar_wait(smem_u32(&pb.empty[st]), eph);
                const uint32_t bar = smem_u32(&pb.full[st]);
                mbar_expect_tx(bar, (uint32_t)(HOPB + BB));
                tma_load_2d(smem_u32(hop_s + (size_t)st * HOPB), &tmap, s * TCOLS, (int)row0, bar);
                bulk_load_1d(smem_u32(b_s + (size_t)st * BB), a.dig + (size_t)s * BB, (uint32_t)BB, bar);
                if (++st == a.stages) { st = 0; eph ^= 1u; }
            }
        }
    }
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem, 512);
    }
}

// ---- backward: dS on the tensor cores, over the rows with a non-zero output gradient only --------------------------------
// dS[j,c] = sum_i sum_d 1[b(hop[i,j]) = d] * TG[i,d,c],  TG[i,d,c] = T[ti,d,c'] * rscale[i,d] * g[i,c].
// A row whose g is entirely zero contributes exactly nothing: a node task trained on a mask (trainer.py:52-58, main.py
// train_mask) has a few hundred such rows out of N, so the rows are compacted first (ordered, deterministic) and only their
// hop bytes are streamed. Layout: a TMEM lane = a hop COLUMN j, the contraction index is (active row, bin slot).

__global__ void row_flags_kernel(const float *__restrict__ g, int64_t R, int C, uint8_t *__restrict__ flags)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R) return;
    bool nz = false;
    for (int c = 0; c < C; ++c) nz |= g[i * C + c] != 0.f;
    flags[i] = nz ? 1 : 0;
}

// one CTA: ordered compaction of the flagged rows -> rows[0..nact), nact
__global__ void __launch_bounds__(1024) compact_rows_kernel(const uint8_t *__restrict__ flags, int64_t R, int32_t *__restrict__ rows,
                                                            int32_t *__restrict__ nact)
{
    __shared__ int wsum[32];
    __shared__ int base_s;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (threadIdx.x == 0) base_s = 0;
    __syncthreads();
    for (int64_t i0 = 0; i0 < R; i0 += 1024) {
        const int64_t i = i0 + threadIdx.x;
        const bool f = i < R && flags[i];
        const unsigned b = __ballot_sync(0xffffffffu, f);
        if (lane == 0) wsum[w] = __popc(b);
        __syncthreads();
        int off = base_s;
        for (int k = 0; k < w; ++k) off += wsum[k];
        if (f) rows[off + __popc(b & ((1u << lane) - 1))] = (int32_t)i;
        __syncthreads();
        if (threadIdx.x == 0) {
            int t = 0;
            for (int k = 0; k < 32; ++k) t += wsum[k];
            base_s += t;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) *nact = base_s;
}

struct TgArgs {
    const float *T, *rscale, *g;
    int per_row, nbins, Cr, C, NB;
    const int32_t *rows, *nact;
};

// value of the B operand at (active row k, bin slot, channel c); slot NB-1 = the unreachable bin, slots in [nbins-1, NB-1) unused
__device__ __forceinline__ float tg_value(const TgArgs &a, int k, int slot, int c)
{
    if (slot >= a.nbins - 1 && slot != a.NB - 1) return 0.f;
    const int d = slot == a.NB - 1 ? a.nbins - 1 : slot;
    const int64_t i = a.rows[k];
    const int cr = a.Cr == 1 ? 0 : c;
    float t = a.per_row ? a.T[(i * a.nbins + d) * a.Cr + cr] : a.T[d * a.Cr + cr];
    if (a.rscale) t *= a.rscale[i * a.nbins + d];
    return t * a.g[i * a.C + c];
}

__global__ void tg_colmax_kernel(TgArgs a, uint32_t *__restrict__ colmax)
{
    const int nact = *a.nact;
    const int64_t total = (int64_t)nact * a.NB, stride = (int64_t)gridDim.x * blockDim.x;
    for (int c = 0; c < a.C; ++c) {
        uint32_t m = 0;
        for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += stride)
            m = max(m, __float_as_uint(fabsf(tg_value(a, (int)(t / a.NB), (int)(t % a.NB), c))));
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, s));
        if ((threadIdx.x & 31) == 0 && m) atomicMax(colmax + c, m);
    }
}

// digit matrix of TG: block = one pipeline stage = 128/NB active rows x NB slots = 128 contraction indices
__global__ void tg_digits_kernel(TgArgs a, const uint32_t *__restrict__ colmax, int ndig, int cpc, int NP, int8_t *__restrict__ dig,
                                 int32_t *__restrict__ colsh)
{
    const int blk = blockIdx.x, nact = *a.nact, RS = TCOLS / a.NB;
    if (blk == 0 && threadIdx.x < a.C) colsh[threadIdx.x] = digit_shift(colmax[threadIdx.x], ndig);
    if (blk * RS >= nact) return;
    for (int t = threadIdx.x; t < NP * TCOLS; t += blockDim.x) {
        const int n = t / TCOLS, k = t % TCOLS;
        const int kk = blk * RS + k / a.NB, slot = k % a.NB;
        const int chunk = n >> 4, w = n & 15, cc = w / ndig, kd = w % ndig;
        const int c = chunk * cpc + cc;
        int8_t v = 0;
        if (kk < nact && cc < cpc && c < a.C) {
            long long q = __double2ll_rn(ldexp((double)tg_value(a, kk, slot, c), digit_shift(colmax[c], ndig)));
            for (int s = 0; s < kd; ++s) {
                const long long b = ((q + 128) & 255) - 128;
                q = (q - b) >> 8;
            }
            v = kd == ndig - 1 ? (int8_t)q : (int8_t)(((q + 128) & 255) - 128);
        }
        dig[(size_t)blk * NP * TCOLS + digit_offset(n, k)] = v;
    }
}

struct DsTcArgs {
    const uint8_t *hop;
    int64_t N, ld;
    int C, ndig, cpc, NP, stages;
    const int32_t *rows, *nact, *colsh;
    const int8_t *dig;
    float *out;       // [gridDim.y][N][C] partial sums (or dS itself when gridDim.y == 1)
};

// one hop byte -> its NB one-hot int8 values (NB/4 TMEM columns)
// `one` = 1 held in ONE register by the caller (an immediate would be re-materialised per prmt)
template <int NB>
__device__ __forceinline__ void onehot_row(uint32_t h, uint32_t *v, uint32_t one)
{
    if (NB == 8) {
        const uint32_t H = (h & 7u) * 0x1111u;
        v[0] = prmt(one, 0u, H ^ 0x3210u); v[1] = prmt(one, 0u, H ^ 0x7654u);
    } else if (NB == 16) {
        const uint32_t H = (h & 15u) * 0x1111u;
        v[0] = prmt(one, 0u, H ^ 0x3210u); v[1] = prmt(one, 0u, H ^ 0x7654u);
        v[2] = prmt(one, 0u, H ^ 0xba98u); v[3] = prmt(one, 0u, H ^ 0xfedcu);
    } else {
        const uint32_t hh = h & 31u, H = (hh & 7u) * 0x1111u, q = hh >> 3;
        const uint32_t p0 = prmt(one, 0u, H ^ 0x3210u), p1 = prmt(one, 0u, H ^ 0x7654u);
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            v[2 * w] = q == (uint32_t)w ? p0 : 0u;
            v[2 * w + 1] = q == (uint32_t)w ? p1 : 0u;
        }
    }
}

// grid (column blocks of NGR*128, row super-blocks); the active-row list is split evenly over the super-blocks
template <int NB, int NGR>
__global__ void __launch_bounds__(TcCfg<NB, NGR>::THREADS, 1)
agg_tc_ds_kernel(DsTcArgs a)
{
    using Cfg = TcCfg<NB, NGR>;
    constexpr int RS = 128 / NB;                 // active hop rows per stage (RS * NB = 128 contraction indices)
    constexpr int CW = NGR * 128;                // hop columns per CTA
    constexpr int HOPB = RS * CW;
    extern __shared__ __align__(1024) uint8_t smem[];
    const int BB = a.NP * TCOLS;
    uint8_t *hop_s = smem;
    uint8_t *b_s = hop_s + (size_t)a.stages * HOPB;
    const PipeBars pb = carve_bars<NGR>(b_s + (size_t)a.stages * BB);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nact = *a.nact;
    const int per = (((nact + (int)gridDim.y - 1) / (int)gridDim.y + RS - 1) / RS) * RS;
    const int k0 = (int)blockIdx.y * per, k1 = min(nact, k0 + per);
    const int nst = k1 > k0 ? (k1 - k0 + RS - 1) / RS : 0;
    const int64_t col0 = (int64_t)blockIdx.x * CW;
    const uint32_t wbytes = (uint32_t)min((int64_t)CW, a.ld - col0);      // ld % 16 == 0: a multiple of 16
    const uint32_t tmem = pipe_setup<NGR>(pb, a.stages);

    if (warp < NGR * 4) {
        // ===== generators: thread m of group g owns TMEM lane m = hop column col0 + g*128 + m =====
        const int g = warp >> 2, m = tid & 127;
        const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
        const uint8_t *hcol = hop_s + g * 128 + m;
        int st = 0, buf = 0;
        uint32_t fph = 0, eph = 1;
        uint32_t h[RS], one;
        asm volatile("mov.u32 %0, 1;" : "=r"(one));
        if (nst > 0) {
            mbar_wait(smem_u32(&pb.full[0]), 0);
#pragma unroll
            for (int r = 0; r < RS; ++r) h[r] = hcol[r * CW];
        }
        for (int s = 0; s < nst; ++s) {
            uint32_t v[32];
#pragma unroll
            for (int r = 0; r < RS; ++r) onehot_row<NB>(h[r], &v[r * (NB / 4)], one);
            mbar_wait(smem_u32(&pb.a_empty[g * NBUF + buf]), eph);
            tc_fence_after();
            tmem_st32(lane_base + (uint32_t)((g * NBUF + buf) * 32), v);
            const int cur = buf;
            if (++st == a.stages) { st = 0; fph ^= 1u; }
            if (++buf == NBUF) { buf = 0; eph ^= 1u; }
            if (s + 1 < nst) {                                        // the next stage's bytes load while the TMEM store lands
                mbar_wait(smem_u32(&pb.full[st]), fph);
                const uint8_t *hs = hcol + (size_t)st * HOPB;
#pragma unroll
                for (int r = 0; r < RS; ++r) h[r] = hs[r * CW];
            }
            tmem_wait_st();
            tc_fence_before();
            mbar_arrive(smem_u32(&pb.a_full[g * NBUF + cur]));
        }
        const int64_t j = col0 + g * 128 + m;
        float *dst = a.out + ((size_t)blockIdx.y * a.N + (j < a.N ? j : 0)) * a.C;
        if (nst > 0) {
            mbar_wait(smem_u32(&pb.acc_full[g]), 0);
            tc_fence_after();
        }
        for (int n0 = 0; n0 < a.NP; n0 += 16) {
            uint32_t acc[16];
            if (nst > 0) {
                tmem_ld16(lane_base + (uint32_t)(Cfg::ACC0 + g * a.NP + n0), acc);
                tmem_wait_ld();
            } else {
#pragma unroll
                for (int q = 0; q < 16; ++q) acc[q] = 0u;
            }
#pragma unroll
            for (int cc = 0; cc < 5; ++cc) {
                const int c = (n0 >> 4) * a.cpc + cc;
                if (cc >= a.cpc || c >= a.C) break;
                long long tot = 0;
                if (a.ndig == 4) {
#pragma unroll
                    for (int k = 3; k >= 0; --k) tot = tot * 256 + (int)acc[(cc * 4 + k) & 15];
                } else {
#pragma unroll
                    for (int k = 2; k >= 0; --k) tot = tot * 256 + (int)acc[(cc * 3 + k) & 15];
                }
                if (j < a.N) dst[c] = (float)ldexp((double)tot, -a.colsh[c]);
            }
        }
        tc_fence_before();
    } else if (warp < NGR * 5) {
        issuer_loop<NGR>(pb, tmem, warp - NGR * 4, lane, nst, a.stages, a.NP, Cfg::ACC0, b_s, BB);
    } else {
        // ===== producer warp: lane r gathers active row r of the stage with one bulk copy (the row indices are read coalesced,
        // one stage ahead), lane 31 brings the digit block =====
        int st = 0;
        uint32_t eph = 1;
        int64_t row = (lane < RS && k0 + lane < k1) ? (int64_t)a.rows[k0 + lane] : 0;
        for (int s = 0; s < nst; ++s) {
            const int kb = k0 + s * RS, nr = min(RS, k1 - kb);
            const int kn = kb + RS + lane;
            const int64_t row_next = (lane < RS && kn < k1) ? (int64_t)a.rows[kn] : 0;
            mbar_wait(smem_u32(&pb.empty[st]), eph);
            const uint32_t bar = smem_u32(&pb.full[st]);
            if (lane == 0) mbar_expect_tx(bar, (uint32_t)nr * wbytes + (uint32_t)BB);
            __syncwarp();
            if (lane < nr) bulk_load_1d(smem_u32(hop_s + (size_t)st * HOPB + lane * CW), a.hop + row * a.ld + col0, wbytes, bar);
            if (lane == 31) bulk_load_1d(smem_u32(b_s + (size_t)st * BB), a.dig + (size_t)(kb / RS) * BB, (uint32_t)BB, bar);
            row = row_next;
            if (++st == a.stages) { st = 0; eph ^= 1u; }
        }
    }
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem, 512);
    }
}

// ---- host side -------------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn()
{
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// uint8 [rows, ld] matrix, box = [box_rows x 128 bytes]; out-of-range elements read as 0
int make_hop_tmap(CUtensorMap *map, const uint8_t *hop, int64_t rows, int64_t ld, int box_rows)
{
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) {
        gnan_set_error("aggregate_rows (tensor-core path): cuTensorMapEncodeTiled is not available from this driver");
        return GNAN_ERR_CUDA;
    }
    const cuuint64_t gdim[2] = {(cuuint64_t)ld, (cuuint64_t)rows};
    const cuuint64_t gstride[1] = {(cuuint64_t)ld};
    const cuuint32_t box[2] = {(cuuint32_t)TCOLS, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult rc = fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<uint8_t *>(hop), gdim, gstride, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (rc != CUDA_SUCCESS) {
        gnan_set_error("aggregate_rows (tensor-core path): cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld ld=%lld)", (int)rc,
                       (long long)rows, (long long)ld);
        return GNAN_ERR_CUDA;
    }
    return GNAN_OK;
}

inline size_t align256(size_t x) { return (x + 255) / 256 * 256; }

// generator groups per CTA: every group owns NBUF A buffers (32 TMEM columns each) and NP accumulator columns of the 512
inline int groups_for(int NP) { return std::max(1, std::min(4, 512 / (NBUF * 32 + NP))); }

struct FwdWs { uint32_t *colmax; int32_t *colsh; int8_t *dig; size_t total; };
FwdWs fwd_ws_layout(void *base, int64_t N, int C)
{
    const DigitPlan p = digit_plan(C);
    const int64_t nblk = ceil_div64(N, TCOLS);
    FwdWs w;
    uint8_t *b = (uint8_t *)base;
    w.colmax = (uint32_t *)b;
    w.colsh = (int32_t *)(b + align256(sizeof(uint32_t) * C));
    w.dig = (int8_t *)(b + 2 * align256(sizeof(uint32_t) * C));
    w.total = 2 * align256(sizeof(uint32_t) * C) + (size_t)nblk * p.NP * TCOLS;
    return w;
}

template <int NB, int NGR>
int launch_fwd(const CUtensorMap &map, AggTcArgs a, cudaStream_t st)
{
    using Cfg = TcCfg<NB, NGR>;
    const size_t per_stage = (size_t)Cfg::HOPB + (size_t)a.NP * TCOLS;
    const size_t fixed = sizeof(uint32_t) * NGR * Cfg::NIB_WORDS + pipe_bar_bytes(NGR);
    int stages = (int)std::min<size_t>(MAX_STAGES, (200 * 1024 - fixed) / per_stage);
    if (stages < 2) {
        gnan_set_error("aggregate_rows (tensor-core path): stage of %zu bytes does not fit shared memory", per_stage);
        return GNAN_ERR_UNSUPPORTED;
    }
    stages = std::min(stages, std::max(2, a.nblk));
    a.stages = stages;
    const size_t smem = fixed + per_stage * stages;
    GNAN_CUDA(cudaFuncSetAttribute(agg_tc_fwd_kernel<NB, NGR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const unsigned grid = (unsigned)ceil_div64(a.R, Cfg::ROWS);
    agg_tc_fwd_kernel<NB, NGR><<<grid, Cfg::THREADS, smem, st>>>(map, a);
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}

template <int NB>
int launch_fwd_nb(const CUtensorMap &map, const AggTcArgs &a, int ngr, cudaStream_t st)
{
    if (ngr == 4) return launch_fwd<NB, 4>(map, a, st);
    if (ngr == 3) return launch_fwd<NB, 3>(map, a, st);
    if (ngr == 2) return launch_fwd<NB, 2>(map, a, st);
    return launch_fwd<NB, 1>(map, a, st);
}

// lanes per row = the bins actually present (even count 10 / 12 / 14): only instantiated for the tensor-bound shapes (NGR <= 3)
template <int NB>
int launch_fwd_exact(const CUtensorMap &map, const AggTcArgs &a, int ngr, cudaStream_t st)
{
    if (ngr == 3) return launch_fwd<NB, 3>(map, a, st);
    if (ngr == 2) return launch_fwd<NB, 2>(map, a, st);
    return launch_fwd<NB, 1>(map, a, st);
}

// lanes per hop row of the forward kernel. With >= 64 digit columns (C >= 13) the pass is bound by the int8 tensor pipe and the
// bins that do not exist are pure waste: a 12-bin table (ogbn-arxiv shape) then puts 10 instead of 8 rows into every MMA.
inline int fwd_lanes_per_row(int nbins, int NP)
{
    if (nbins <= 8) return 8;
    if (nbins > 16) return 32;
    const int even = (nbins + 1) & ~1;
    return (NP >= 64 && even < 16) ? even : 16;
}

// true when the tensor-core path covers the shape (nbins <= 32, accumulator columns <= 256, a matrix worth a TMA pipeline)
bool tc_supported(int64_t R, int64_t N, int64_t ld_hop, int32_t nbins, int32_t C)
{
    if (R < 1 || N < 256 || ld_hop < TCOLS || nbins < 2 || nbins > 32 || C < 1) return false;
    return digit_plan(C).NP <= 256;
}

}  // namespace

// CUDA-core path (agg.cu)
int gnan_agg_rows_fwd_cuda_cores(const uint8_t *hop, int64_t R, int64_t N, int64_t ld_hop, const float *T, int table_per_row,
                                 int32_t nbins, int32_t Cr, const float *rscale, const float *S, int32_t C, float *out, float *Bsum,
                                 gnan_stream_t stream);
size_t gnan_agg_rows_bwd_cuda_cores_bytes(int64_t R, int64_t N, int32_t nbins, int32_t C);
int gnan_agg_rows_bwd_cuda_cores(const uint8_t *hop, int64_t R, int64_t N, int64_t ld_hop, const float *T, int table_per_row,
                                 int32_t nbins, int32_t Cr, const float *rscale, const float *S, int32_t C, const float *g,
                                 const float *Bsum, float *dS, float *dT, void *workspace, size_t workspace_bytes,
                                 gnan_stream_t stream);

extern "C" size_t gnan_aggregate_rows_fwd_workspace_bytes(int64_t R, int64_t N, int64_t ld_hop, int32_t nbins, int32_t C)
{
    if (!tc_supported(R, N, ld_hop, nbins, C)) return 0;
    return fwd_ws_layout(nullptr, N, C).total;
}

extern "C" int gnan_aggregate_rows_fwd_ws(const uint8_t *hop, int64_t R, int64_t N, int64_t ld_hop, const float *T,
                                          int table_per_row, int32_t nbins, int32_t Cr, const float *rscale, const float *S,
                                          int32_t C, float *out, float *Bsum, int algo, void *workspace, size_t workspace_bytes,
                                          gnan_stream_t stream)
{
    const bool can_tc = tc_supported(R, N, ld_hop, nbins, C);
    // auto: with a single channel the CUDA-core bin sums stream the hop bytes faster (measured 1.6 TB/s vs 1.0 TB/s at the
    // ogbn-arxiv shape); from two channels on they re-stream per channel chunk and the tensor-core pass wins
    if (algo == GNAN_AGG_CUDA_CORES || (algo == GNAN_AGG_AUTO && (!can_tc || C < 2)))
        return gnan_agg_rows_fwd_cuda_cores(hop, R, N, ld_hop, T, table_per_row, nbins, Cr, rscale, S, C, out, Bsum, stream);
    GNAN_REQUIRE(algo == GNAN_AGG_AUTO || algo == GNAN_AGG_TENSOR_CORES, "aggregate_rows_fwd_ws: unknown algo %d", algo);
    if (!can_tc) {
        gnan_set_error("aggregate_rows_fwd_ws: the tensor-core path needs N >= 256, nbins <= 32 and <= 256 accumulator columns "
                       "(N=%lld nbins=%d C=%d)", (long long)N, nbins, C);
        return GNAN_ERR_UNSUPPORTED;
    }
    GNAN_REQUIRE(hop && T && S && out, "aggregate_rows_fwd_ws: NULL hop/T/S/out");
    GNAN_REQUIRE(ld_hop >= N && ld_hop % 16 == 0 && ((uintptr_t)hop % 16) == 0, "aggregate_rows_fwd_ws: hop rows must be 16-byte aligned with ld %% 16 == 0");
    GNAN_REQUIRE(Cr == 1 || Cr == C, "aggregate_rows_fwd_ws: Cr must be 1 or C");
    const FwdWs w = fwd_ws_layout(workspace, N, C);
    if (!workspace || workspace_bytes < w.total) {
        gnan_set_error("aggregate_rows_fwd_ws: workspace %zu < %zu bytes", workspace_bytes, w.total);
        return GNAN_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const DigitPlan p = digit_plan(C);
    const int nblk = (int)ceil_div64(N, TCOLS);
    GNAN_CUDA(cudaMemsetAsync(w.colmax, 0, sizeof(uint32_t) * C, st));
    colmax_kernel<<<(unsigned)std::min<int64_t>(ceil_div64(N, 256), 4 * gnan_sm_count()), 256, 0, st>>>(S, N, C, w.colmax);
    GNAN_LAUNCH_OK();
    digits_kernel<<<nblk, 256, 0, st>>>(S, N, C, C, nullptr, w.colmax, p.ndig, p.cpc, p.NP, w.dig, w.colsh);
    GNAN_LAUNCH_OK();

    AggTcArgs a{R, N, nbins, C, Cr, table_per_row, p.ndig, p.cpc, p.NP, nblk, 0, T, rscale, w.colsh, w.dig, out, Bsum};
    const int ngr = groups_for(p.NP);
    const int nb = fwd_lanes_per_row(nbins, p.NP);
    CUtensorMap map;
    int rc = make_hop_tmap(&map, hop, R, ld_hop, (128 / nb) * ngr);
    if (rc) return rc;
    if (nb == 8) return launch_fwd_nb<8>(map, a, ngr, st);
    if (nb == 10) return launch_fwd_exact<10>(map, a, ngr, st);
    if (nb == 12) return launch_fwd_exact<12>(map, a, ngr, st);
    if (nb == 14) return launch_fwd_exact<14>(map, a, ngr, st);
    if (nb == 16) return launch_fwd_nb<16>(map, a, ngr, st);
    return launch_fwd_nb<32>(map, a, ngr, st);
}

// ---- backward host side -------------------------------------------------------------------------------------------------------
namespace {

struct BwdPlan { int nb, ngr, RS, CW, ncol, nsb; DigitPlan dp; };
// The backward always carries FOUR digits when they fit: the rounding error of TG[i,d,c] is shared by every column j with
// b(hop[i,j]) = d, so a weight gradient (a sum of dS over thousands of columns: d bo = sum_j dS[j]) sees it amplified by the
// level size. Measured with 3 digits (C = 5, 4000 nodes): 1.4e-4 on the shape-function gradients; with 4 digits 1e-7.
inline DigitPlan digit_plan_bwd(int C)
{
    const int c4 = (C + 3) / 4;
    if (16 * c4 > 256) return digit_plan(C);
    DigitPlan p;
    p.ndig = 4; p.cpc = 4; p.NP = 16 * c4;
    return p;
}

BwdPlan bwd_plan(int64_t R, int64_t N, int nbins, int C)
{
    BwdPlan p;
    p.dp = digit_plan_bwd(C);
    p.nb = nbins <= 8 ? 8 : (nbins <= 16 ? 16 : 32);
    p.ngr = groups_for(p.dp.NP);
    p.RS = 128 / p.nb;
    p.CW = p.ngr * 128;
    p.ncol = (int)ceil_div64(N, p.CW);
    int nsb = (int)ceil_div64(2 * gnan_sm_count(), p.ncol);
    const int64_t max_sb = std::max<int64_t>(1, ceil_div64(R, 4 * p.RS));       // at least 4 stages per super-block when all rows are active
    p.nsb = (int)std::max<int64_t>(1, std::min<int64_t>(nsb, max_sb));
    return p;
}

struct BwdWs { uint8_t *flags; int32_t *rows, *nact; uint32_t *colmax; int32_t *colsh; int8_t *dig; float *part; size_t total; };
BwdWs bwd_ws_layout(void *base, int64_t R, int64_t N, int C, const BwdPlan &p)
{
    BwdWs w;
    uint8_t *b = (uint8_t *)base;
    size_t o = 0;
    w.flags = b + o; o += align256((size_t)R);
    w.rows = (int32_t *)(b + o); o += align256(sizeof(int32_t) * (size_t)R);
    w.nact = (int32_t *)(b + o); o += 256;
    w.colmax = (uint32_t *)(b + o); o += align256(sizeof(uint32_t) * C);
    w.colsh = (int32_t *)(b + o); o += align256(sizeof(int32_t) * C);
    w.dig = (int8_t *)(b + o); o += (size_t)ceil_div64(R, p.RS) * p.dp.NP * TCOLS;
    w.part = (float *)(b + o); o += p.nsb > 1 ? sizeof(float) * (size_t)p.nsb * N * C : 0;
    w.total = o;
    return w;
}

template <int NB, int NGR>
int launch_ds(DsTcArgs a, int ncol, int nsb, cudaStream_t st)
{
    using Cfg = TcCfg<NB, NGR>;
    const size_t per_stage = (size_t)(128 / NB) * NGR * 128 + (size_t)a.NP * TCOLS;
    const size_t fixed = pipe_bar_bytes(NGR);
    int stages = (int)std::min<size_t>(MAX_STAGES, (200 * 1024 - fixed) / per_stage);
    if (stages < 2) {
        gnan_set_error("aggregate_rows_bwd (tensor-core path): stage of %zu bytes does not fit shared memory", per_stage);
        return GNAN_ERR_UNSUPPORTED;
    }
    a.stages = stages;
    const size_t smem = fixed + per_stage * stages;
    GNAN_CUDA(cudaFuncSetAttribute(agg_tc_ds_kernel<NB, NGR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    agg_tc_ds_kernel<NB, NGR><<<dim3((unsigned)ncol, (unsigned)nsb), Cfg::THREADS, smem, st>>>(a);
    GNAN_LAUNCH_OK();
    return GNAN_OK;
}

template <int NB>
int launch_ds_nb(const DsTcArgs &a, const BwdPlan &p, cudaStream_t st)
{
    if (p.ngr == 4) return launch_ds<NB, 4>(a, p.ncol, p.nsb, st);
    if (p.ngr == 3) return launch_ds<NB, 3>(a, p.ncol, p.nsb, st);
    if (p.ngr == 2) return launch_ds<NB, 2>(a, p.ncol, p.nsb, st);
    return launch_ds<NB, 1>(a, p.ncol, p.nsb, st);
}

}  // namespace

extern "C" size_t gnan_aggregate_rows_bwd_ws_bytes(int64_t R, int64_t N, int64_t ld_hop, int32_t nbins, int32_t Cr, int32_t C, int algo)
{
    if (algo == GNAN_AGG_CUDA_CORES || !tc_supported(R, N, ld_hop, nbins, C))
        return gnan_agg_rows_bwd_cuda_cores_bytes(R, N, nbins, C);
    const BwdPlan p = bwd_plan(R, N, nbins, C);
    return bwd_ws_layout(nullptr, R, N, C, p).total;       // dT needs no workspace when the bin sums were saved
}

extern "C" int gnan_aggregate_rows_bwd_ws(const uint8_t *hop, int64_t R, int64_t N, int64_t ld_hop, const float *T,
                                          int table_per_row, int32_t nbins, int32_t Cr, const float *rscale, const float *S,
                                          int32_t C, const float *g, const float *Bsum, float *dS, float *dT, int algo,
                                          void *workspace, size_t workspace_bytes, gnan_stream_t stream)
{
    const bool can_tc = tc_supported(R, N, ld_hop, nbins, C) && Bsum != nullptr;
    if (algo == GNAN_AGG_CUDA_CORES || (algo == GNAN_AGG_AUTO && !can_tc))
        return gnan_agg_rows_bwd_cuda_cores(hop, R, N, ld_hop, T, table_per_row, nbins, Cr, rscale, S, C, g, Bsum, dS, dT, workspace,
                                            workspace_bytes, stream);
    GNAN_REQUIRE(algo == GNAN_AGG_AUTO || algo == GNAN_AGG_TENSOR_CORES, "aggregate_rows_bwd_ws: unknown algo %d", algo);
    if (!can_tc) {
        gnan_set_error("aggregate_rows_bwd_ws: the tensor-core path needs saved bin sums, N >= 256, nbins <= 32 and <= 256 accumulator "
                       "columns (N=%lld nbins=%d C=%d)", (long long)N, nbins, C);
        return GNAN_ERR_UNSUPPORTED;
    }
    GNAN_REQUIRE(hop && T && S && g, "aggregate_rows_bwd_ws: NULL hop/T/S/g");
    GNAN_REQUIRE(ld_hop >= N && ld_hop % 16 == 0 && ((uintptr_t)hop % 16) == 0, "aggregate_rows_bwd_ws: hop rows must be 16-byte aligned with ld %% 16 == 0");
    GNAN_REQUIRE(R < (int64_t)1 << 31, "aggregate_rows_bwd_ws: too many rows");
    cudaStream_t st = (cudaStream_t)stream;
    if (dT) {   // from the saved bin sums, no pass over the hop block (the CUDA-core helper with dS = NULL)
        int rc = gnan_agg_rows_bwd_cuda_cores(hop, R, N, ld_hop, T, table_per_row, nbins, Cr, rscale, S, C, g, Bsum, nullptr, dT, nullptr, 0, stream);
        if (rc) return rc;
    }
    if (!dS) return GNAN_OK;
    const BwdPlan p = bwd_plan(R, N, nbins, C);
    const BwdWs w = bwd_ws_layout(workspace, R, N, C, p);
    if (!workspace || workspace_bytes < w.total) {
        gnan_set_error("aggregate_rows_bwd_ws: workspace %zu < %zu bytes", workspace_bytes, w.total);
        return GNAN_ERR_WORKSPACE;
    }
    row_flags_kernel<<<(unsigned)ceil_div64(R, 256), 256, 0, st>>>(g, R, C, w.flags);
    GNAN_LAUNCH_OK();
    compact_rows_kernel<<<1, 1024, 0, st>>>(w.flags, R, w.rows, w.nact);
    GNAN_LAUNCH_OK();
    GNAN_CUDA(cudaMemsetAsync(w.colmax, 0, sizeof(uint32_t) * C, st));
    TgArgs ta{T, rscale, g, table_per_row, nbins, Cr, C, p.nb, w.rows, w.nact};
    tg_colmax_kernel<<<(unsigned)std::min<int64_t>(ceil_div64(R * p.nb, 256), 2 * gnan_sm_count()), 256, 0, st>>>(ta, w.colmax);
    GNAN_LAUNCH_OK();
    tg_digits_kernel<<<(unsigned)ceil_div64(R, p.RS), 256, 0, st>>>(ta, w.colmax, p.dp.ndig, p.dp.cpc, p.dp.NP, w.dig, w.colsh);
    GNAN_LAUNCH_OK();
    DsTcArgs a{hop, N, ld_hop, C, p.dp.ndig, p.dp.cpc, p.dp.NP, 0, w.rows, w.nact, w.colsh, w.dig, p.nsb > 1 ? w.part : dS};
    int rc = p.nb == 8 ? launch_ds_nb<8>(a, p, st) : (p.nb == 16 ? launch_ds_nb<16>(a, p, st) : launch_ds_nb<32>(a, p, st));
    if (rc) return rc;
    if (p.nsb > 1) {
        const size_t n = (size_t)N * C;
        rc = gnan_reduce_chunks(w.part, p.nsb, n, n, dS, st);
    }
    return rc;
}
