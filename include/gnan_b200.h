/*
 * gnan_b200 — C ABI of the B200 (sm_100a) GNAN hot path.
 *
 * The reference (mayabechlerspeicher/Graph-Neural-Additive-Networks---GNAN) is pure Python/PyTorch and
 * defines no FFI of its own (SURVEY.md §8b): the "plugin boundary" upstream is the nn.Module. This header
 * is the boundary a maintainer binds instead of the stock ATen ops the reference modules run; each entry
 * point names the reference lines it replaces. INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; the caller (PyTorch) owns all
 *     memory, the library never allocates, frees or retains a pointer;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing synchronises;
 *   - return value: GNAN_OK or an error code; gnan_last_error() returns a thread-local message;
 *   - float tensors are contiguous fp32 row-major unless a leading dimension is given;
 *   - no CPU fallback: a call on a machine without an sm_100 device fails with GNAN_ERR_CUDA.
 */
#ifndef GNAN_B200_H
#define GNAN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GNAN_B200_VERSION 102

enum {
    GNAN_OK = 0,
    GNAN_ERR_INVALID = 1,     /* bad argument (shape, alignment, null pointer) */
    GNAN_ERR_UNSUPPORTED = 2, /* valid but not implemented for this shape (e.g. hidden width) */
    GNAN_ERR_CUDA = 3,        /* a CUDA runtime call failed; message has cudaGetErrorString */
    GNAN_ERR_WORKSPACE = 4    /* workspace too small; query the matching *_workspace_bytes */
};

#define GNAN_HOP_UNREACHABLE 255 /* byte value of an unreachable / masked pair in a hop matrix */
#define GNAN_APSP_BATCHED_MAX_NODES 1024 /* largest graph of gnan_apsp_bfs_batched_ex */

typedef void *gnan_stream_t;

int gnan_version(void);
const char *gnan_last_error(void);
/* number of kernels this library has launched in the calling process (bench.py's gpu_launches evidence) */
uint64_t gnan_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * Grouped scalar-input MLPs: G independent networks  R -> R^C,
 *     Linear(1,H) ReLU [Dropout]  ( Linear(H,H) ReLU [Dropout] ) x n_hidden   Linear(H,C)
 * n_layers = n_hidden + 2;  n_layers == 1 is the single Linear(1,C) (w1/b1/wh/bh unused, H ignored).
 * Used for the K shape functions f_k (G = K, GNAN.py:24-34, models.py:321-331) and, with G = 1 and no
 * dropout, for the distance function rho evaluated on a table of inputs (GNAN.py:38-47).
 * Weight layout = torch.nn.Linear's [out,in], stacked over groups. Bias pointers may be NULL (bias=False).
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t G, H, C, n_layers;
    const float *w1; /* [G,H]            Linear(1,H).weight[:,0] */
    const float *b1; /* [G,H] or NULL */
    const float *wh; /* [n_hidden,G,H,H] */
    const float *bh; /* [n_hidden,G,H] or NULL */
    const float *wo; /* [G,C,H]  ([G,C,1] when n_layers == 1) */
    const float *bo; /* [G,C] or NULL */
} gnan_mlp_params;

typedef struct { /* gradient outputs, same shapes; NULL = not wanted. Overwritten, not accumulated. */
    float *w1, *b1, *wh, *bh, *wo, *bo;
    float *du; /* [R,G] gradient w.r.t. the scalar inputs u, or NULL. Only the NAM readout needs it (its inputs are the
                  pooled per-feature values, models.py:379-381); requesting it selects the fp32 kernels. */
} gnan_mlp_grads;

/* precision: how the HxH hidden contractions are computed */
enum {
    GNAN_PREC_FP32 = 0,     /* FFMA, fp32 throughout (bit-for-bit deterministic) */
    GNAN_PREC_TF32X3 = 1,   /* tcgen05 kind::tf32, 3-term split (hi*hi + lo*hi + hi*lo), fp32 accumulate in TMEM:
                               fp32-level accuracy (~1e-6 norm-wise); needs H == 64 */
    GNAN_PREC_TF32 = 2      /* tcgen05 single-pass tf32 (~1e-3), stated looser bound */
};                          /* shapes the tensor-core path does not cover (H != 64, n_layers != 3, C > 64) run the fp32 kernel;
                               gnan_mlp_bwd with 8 < C <= 64 makes ceil(C/8) passes over 8-channel slices (or see gnan_mlp_bwd_ext) */

size_t gnan_mlp_workspace_bytes(int64_t R, const gnan_mlp_params *p, int backward, int precision);

/* S[r,:] = sum_g f_g(u[r*ldu + g])   (replaces the K-iteration module loop + slice assignment + feature sum:
 * GNAN.py:57-62,157; models.py:360-365,455-460; batched_pyg_main.py:144-148,170).
 * dropout_p > 0 applies inverted dropout after every hidden ReLU with a counter-based mask keyed on
 * (seed, layer, group, row, unit); the same (dropout_p, seed, seed_dev) must be passed to gnan_mlp_bwd.
 * seed_dev (optional, NULL = unused): one device-resident 64-bit word XORed into `seed` when the kernel starts. A step that
 * is captured into a CUDA graph bakes by-value arguments in; advancing this word on the device between replays gives every
 * replay fresh masks. */
int gnan_mlp_fwd(const float *u, int64_t R, int64_t ldu, const gnan_mlp_params *p, float dropout_p, uint64_t seed,
                 const uint64_t *seed_dev, int precision, float *S /* [R,C] */, void *workspace, size_t workspace_bytes,
                 gnan_stream_t stream);

/* gradients of all weights given dS [R,C] (replaces autograd through the same lines; trainer.py:66).
 * Activations are recomputed, nothing is saved by the forward. */
int gnan_mlp_bwd(const float *u, int64_t R, int64_t ldu, const gnan_mlp_params *p, float dropout_p, uint64_t seed,
                 const uint64_t *seed_dev, int precision, const float *dS /* [R,C] */, const gnan_mlp_grads *grads,
                 void *workspace, size_t workspace_bytes, gnan_stream_t stream);

/* gnan_mlp_bwd with the OUTPUT LAYER outside the kernel, for more than 8 output channels on the tensor-core path (H = 64, 3
 * layers, precision != fp32): the caller supplies dh [R,G,64] = dS Wo_g (one plain GEMM: [R,C] x [C, G*64]) and receives
 * a1 [R,G,64], the last hidden activation, from which dWo_g = dS^T a1_g is a second plain GEMM; everything else (d bo included)
 * comes back in `grads` (grads->wo and grads->du must be NULL). One pass over the rows for any C instead of ceil(C/8):
 * models.py / GNAN.py shape functions with 40 classes (ogbn-arxiv), GNAN.py:57-62 backward. */
int gnan_mlp_bwd_ext_supported(const gnan_mlp_params *p, int precision);
int gnan_mlp_bwd_ext(const float *u, int64_t R, int64_t ldu, const gnan_mlp_params *p, float dropout_p, uint64_t seed,
                     const uint64_t *seed_dev, int precision, const float *dS, const float *dh /* [R,G,64] */,
                     float *a1 /* [R,G,64] out */, const gnan_mlp_grads *grads, void *workspace, size_t workspace_bytes,
                     gnan_stream_t stream);

/* Entries mode: the shape functions on a COMPRESSED feature matrix (same reference lines as gnan_mlp_fwd/bwd). When
 * dropout is off, rows that carry the same value in a feature column share one evaluation of that feature's MLP (the zeros
 * of a bag-of-words matrix, the off entries of a one-hot encoding, the constant column: datasets.py:94, SURVEY.md §8d).
 * The caller lists the distinct work as val[E] grouped by feature, group g owning entries [grp_ptr[g], grp_ptr[g+1]);
 * Y[e,:] = f_g(val[e]) and the weight gradients given dY[E,C] come back; how entries map to rows of S is the caller's
 * business (gnan_b200/sparse.py). items [n_items,2] = (group, 128-entry tile index inside the group): one CTA per item.
 * Forward: fp32 kernels or, with `precision` != GNAN_PREC_FP32, the tcgen05 kernel for H = 64, 3 layers, C <= 8; backward: fp32
 * or the tcgen05 kernel (`precision`), or — H = 64, 3 layers, C <= 8, at most 96 entries per feature on average and 3 072 in any
 * one — a CTA per feature on the CUDA cores in fp32 under either `precision` (bag-of-words columns: a few dozen entries per
 * feature, where a tensor-core tile would be a quarter full); n_layers >= 2; no dropout (the sharing would be wrong with per-row
 * masks). */
size_t gnan_mlp_entries_workspace_bytes(int64_t max_group_entries, const gnan_mlp_params *p, int backward, int precision);
int gnan_mlp_entries_fwd_ex(const float *val, const int64_t *grp_ptr /* [G+1] */, int64_t E, const int32_t *items, int64_t n_items,
                            const gnan_mlp_params *p, int precision, float *Y /* [E,C] */, gnan_stream_t stream);
int gnan_mlp_entries_bwd(const float *val, const int64_t *grp_ptr, int64_t E, int64_t max_group_entries,
                         const gnan_mlp_params *p, int precision /* backward may run on tcgen05 like gnan_mlp_bwd */,
                         const float *dY /* [E,C] */, const gnan_mlp_grads *grads, void *workspace, size_t workspace_bytes,
                         gnan_stream_t stream);

/* Entry values <-> node rows (deterministic, no atomics). Group g's FIRST entry is the feature's baseline value, shared by
 * every row not listed among its exceptions:  S[r,:] = sum_g Y[base_g,:] + sum_{e in exceptions of row r} (Y[e,:] - Y[base_g(e),:]).
 * csr_ptr/csr_eid list the exception entries of each row, ent_grp[e] / ent_row[e] are an entry's group and row (-1 for a
 * baseline). S0 [C] and dStot [gnan_rows_to_entries_scratch_floats(G,C,E)] are scratch outputs (sum of the baselines; sum of
 * all dS rows in the first C floats, slab partial sums behind). */
size_t gnan_rows_to_entries_scratch_floats(int32_t G, int32_t C, int64_t E);
int gnan_entries_to_rows(const float *Y /* [E,C] */, int64_t N, int32_t G, int32_t C, const int64_t *grp_ptr,
                         const int64_t *csr_ptr /* [N+1] */, const int64_t *csr_eid, const int32_t *ent_grp /* [E] */,
                         float *S0 /* [C] */, float *S /* [N,C] */, gnan_stream_t stream);
int gnan_rows_to_entries(const float *dS /* [N,C] */, int64_t N, int32_t G, int32_t C, const int64_t *grp_ptr, int64_t E,
                         const int64_t *ent_row /* [E] */, float *dStot /* scratch, see above */, float *dY /* [E,C] */, gnan_stream_t stream);

/* out[s,:] = sum_{k in [seg_ptr[s], seg_ptr[s+1])} src[order[k],:]  — the deterministic backward of a row gather T = Tq[inv]
 * (the per-row rho inputs 1/((1+d)*cnt) of GNAN.py:65-67 take few distinct values: rho runs once per distinct value). */
int gnan_gather_segment_sum(const float *src /* [M,C] */, const int64_t *order /* [M], or NULL = rows already in segment order */,
                            const int64_t *seg_ptr /* [nseg+1] */,
                            int64_t nseg, int32_t C, float *out /* [nseg,C] */, gnan_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Distance-table inputs. u[i,d] = 1/(1+d) for d < nbins-1, 0 for the unreachable bin (nbins-1);
 * with cnt != NULL divided by cnt[i,d] (GNAN.py:65-66: node_distances / normalization_matrix).
 * raw != 0 writes u[d] = d instead (batched_pyg_main.py:154: rho is fed raw hop counts).
 * rows == 0 / cnt == NULL -> one global row [nbins].
 * ---------------------------------------------------------------------------------------------- */
int gnan_rho_table_inputs(const int32_t *cnt /* [rows,nbins] or NULL */, int64_t rows, int32_t nbins, int raw,
                          float *u /* [max(rows,1), nbins] */, gnan_stream_t stream);

/* rscale[i,d] = 1/cnt[i,d] (0 where cnt == 0): the output normaliser of models.py:368-370 / GNAN.py:163-168 */
int gnan_level_rscale(const int32_t *cnt, int64_t rows, int32_t nbins, float *rscale, gnan_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Aggregation over a dense row block of the uint8 hop matrix (node-level tasks):
 *     out[i,c] = sum_j  T[ti, b(hop[i,j]), c'] * rscale[i, b(hop[i,j])] * S[j,c]
 * b(h) = h for h <= nbins-2, nbins-1 for h == 255.  c' = c if Cr == C else 0 (Cr == 1: shared rho).
 * table_per_row: T is [R,nbins,Cr] (input-normalised rho, GNAN.py:65-67) else [nbins,Cr]; rscale may be NULL.
 * Replaces GNAN.py:67-73,159-170 and models.py:366-375 (the N*N rho evaluation, permutes, bmm and sums).
 * Both directions go through the per-row bin sums Bsum[i,d,c] = sum_{j: b(hop[i,j]) = d} S[j,c] ([R,nbins,C]).
 *
 * Two kernel families, selected by `algo`:
 *  - CUDA cores (csrc/agg.cu): fp32 bin sums;
 *  - tensor cores (csrc/agg_tc.cu): the reference's matmul(m_dist_perm, fx_perm) (GNAN.py:70, models.py:371-372) as
 *    Bsum[(i,d), c] = sum_j 1[b(hop[i,j]) = d] * S[j,c] on tcgen05 (kind::i8, int32 accumulation in TMEM), the hop tiles
 *    streamed ONCE for all C channels by TMA and the 0/1 operand generated on the fly. S is quantised per channel to 3-4 signed
 *    8-bit digits of a common power-of-two scale (absolute error <= 2^-23 / 2^-31 of the column's largest magnitude); the bin
 *    sums are exact integer sums of the quantised values (order-independent, deterministic), rounded to fp32 once. Covers
 *    N >= 256, nbins <= 32 and <= 256 accumulator columns (C <= 80).
 * ---------------------------------------------------------------------------------------------- */
enum {
    GNAN_AGG_AUTO = 0,         /* tensor cores where the shape is covered, CUDA cores otherwise */
    GNAN_AGG_CUDA_CORES = 1,   /* the fp32 bin-sum kernels of csrc/agg.cu (the forward needs no workspace) */
    GNAN_AGG_TENSOR_CORES = 2  /* fail with GNAN_ERR_UNSUPPORTED when the shape is not covered */
};

/* forward: out [R,C], and Bsum when it is not NULL (the training-mode forward saves it: the backward turns it into dT without
 * another pass over the hop block). The workspace holds the digit matrix of S for the tensor-core path:
 * gnan_aggregate_rows_fwd_workspace_bytes is 0 when that path does not cover the shape, and the CUDA-core path needs none. */
size_t gnan_aggregate_rows_fwd_workspace_bytes(int64_t R, int64_t N, int64_t ld_hop, int32_t nbins, int32_t C);
int gnan_aggregate_rows_fwd_ws(const uint8_t *hop, int64_t R, int64_t N, int64_t ld_hop, const float *T, int table_per_row,
                               int32_t nbins, int32_t Cr, const float *rscale, const float *S, int32_t C, float *out,
                               float *Bsum /* or NULL */, int algo, void *workspace, size_t workspace_bytes,
                               gnan_stream_t stream);

/* backward, given g = dL/dout [R,C]:
 *     dS[j,c] = sum_i W[i,j,c] g[i,c]   (overwritten; [N,C]; NULL = not wanted)
 *     dT (same shape as T; overwritten; NULL = not wanted)  dT[ti,d,c'] = sum_{i in ti} rscale[i,d] * sum_c g[i,c] * Bsum[i,d,c]
 * Bsum is the one the forward saved. With Bsum == NULL the CUDA-core backward recomputes it with one extra pass over the hop
 * block; the tensor-core path needs it (AUTO then runs on the CUDA cores: size the workspace with GNAN_AGG_CUDA_CORES).
 * Tensor-core path: dT from the bin sums; dS[j,c] = sum_{i,d} 1[b(hop[i,j]) = d] * TG[i,d,c] with TG = T*rscale*g quantised
 * like S above, contracted on tcgen05 with a TMEM lane per hop COLUMN. Rows whose g is entirely zero are skipped (their
 * contribution is exactly zero): the hop bytes streamed are those of the rows that carry a loss (a train mask:
 * trainer.py:52-58). Workspace: gnan_aggregate_rows_bwd_ws_bytes with the same `algo`. */
size_t gnan_aggregate_rows_bwd_ws_bytes(int64_t R, int64_t N, int64_t ld_hop, int32_t nbins, int32_t Cr, int32_t C, int algo);
int gnan_aggregate_rows_bwd_ws(const uint8_t *hop, int64_t R, int64_t N, int64_t ld_hop, const float *T, int table_per_row,
                               int32_t nbins, int32_t Cr, const float *rscale, const float *S, int32_t C, const float *g,
                               const float *Bsum, float *dS, float *dT, int algo, void *workspace, size_t workspace_bytes,
                               gnan_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Block-diagonal (batched small graphs) aggregation. Graph b owns nodes [node_off[b], node_off[b+1]) and the
 * packed n_b x n_b hop block at hop + hop_off[b] (row-major, row stride n_b). The dense (sum N)^2 matrix of
 * batched_pyg_main.py:75-80 is never built. reduce_graph != 0 additionally sums over the graph's nodes
 * (GNAN.py:76-78; batched_pyg_main.py:176-181): out is [B,C], else [sum N, C].
 * T / rscale rows are indexed by global node id when table_per_row / rscale are given.
 * ---------------------------------------------------------------------------------------------- */
int gnan_aggregate_blockdiag_fwd(const uint8_t *hop, const int64_t *hop_off /* [B+1] */, const int32_t *node_off /* [B+1] */,
                                 int32_t B, const float *T, int table_per_row, int32_t nbins, int32_t Cr,
                                 const float *rscale, const float *S, int32_t C, int reduce_graph, float *out,
                                 gnan_stream_t stream);

int gnan_aggregate_blockdiag_bwd(const uint8_t *hop, const int64_t *hop_off, const int32_t *node_off, int32_t B,
                                 const float *T, int table_per_row, int32_t nbins, int32_t Cr, const float *rscale,
                                 const float *S, int32_t C, int reduce_graph, const float *g, float *dS,
                                 float *dT /* zero-initialised by the callee; global table grads are atomically added */,
                                 gnan_stream_t stream);

/* Graph-level readout with a GLOBAL table (models.py:366-384 / GNAN.py:64-79 with is_graph_task; batched_pyg_main.py:154-181),
 * csrc/agg_bd.cu: out[b,c] = sum_{i,j in b} T[d_ij,c'] rscale[i,d_ij] S[j,c] is bilinear in (T,S) given the pair statistics
 * P[j,d] = sum_{i: d_ij = d} rscale[i,d]. The forward makes the ONLY pass over the hop bytes and saves
 * colw[j,c'] = sum_d T[d,c'] P[j,d] ([sumN,Cr]) and Q[b,d,c] = sum_j S[j,c] P[j,d] ([B,nbins,C]); the backward is
 * dS[j,c] = g[b,c] colw[j,c'], dT[d,c'] = sum_{b,c} g[b,c] Q[b,d,c] (both overwritten), without touching the hop bytes.
 * Covers nbins <= 64, C <= 4 (see _supported); work_counter: one device int32 (zeroed by the callee; graphs are handed out
 * to the warps dynamically). Deterministic. */
int gnan_aggregate_blockdiag_graph_supported(int32_t nbins, int32_t Cr, int32_t C);
int gnan_aggregate_blockdiag_graph_fwd(const uint8_t *hop, const int64_t *hop_off, const int32_t *node_off, int32_t B,
                                       const float *T /* [nbins,Cr] */, int32_t nbins, int32_t Cr,
                                       const float *rscale /* [sumN,nbins] or NULL */, const float *S, int32_t C,
                                       float *out /* [B,C] */, float *colw, float *Q, int32_t *work_counter, gnan_stream_t stream);
size_t gnan_aggregate_blockdiag_graph_bwd_workspace_bytes(int32_t nbins, int32_t C);
int gnan_aggregate_blockdiag_graph_bwd(const int32_t *node_off, int32_t B, int32_t nbins, int32_t Cr, int32_t C,
                                       const float *g /* [B,C] */, const float *colw, const float *Q, float *dS, float *dT,
                                       void *workspace, size_t workspace_bytes, gnan_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Explanations (csrc/explain.cu; gnan_b200.interpret.explain): the contribution of each shape function k to an output row, the
 * reference's mf = matmul(W, fx) of GNAN.py:68-70 before its sum over features, with W[i,j,c'] = T[t_i, b(hop[i,j]), c'] *
 * rscale[i, b(hop[i,j])] as in gnan_aggregate_rows_fwd_ws. The features come in the compressed form of gnan_mlp_entries_*:
 * group k = [baseline entry, exceptions sorted by row], Y [E,C] the entry values f_k(val[e]), ent_row [E] (-1 for a baseline).
 * Graph b owns nodes [node_off[b], node_off[b+1]) (a dense single graph: B = 1, node_off = {0, N}).
 * seg [K, B+1] (gnan_explain_segments): seg[k,b] = first exception of k with a row >= node_off[b], so the exceptions of feature k
 * inside graph b are [seg[k,b], seg[k,b+1]).
 * Graph rows:  F[b,k,c] = Y[base_k,c] * colw_sum[b,c] + sum_{e in seg(k,b)} colw[row(e),c] * (Y[e,c] - Y[base_k,c])   [B,K,C]
 *   colw [N,C] = sum_{i in graph(j)} W[i,j,c'] (the aggregation's dS for a unit output gradient), colw_sum [B,C] its sum per graph.
 * Node rows:   F[r,k,c] = Y[base_k,c] * sum_j W[i,j,c'] + sum_{e in seg(k,b(i))} W[i,row(e),c'] * (Y[e,c] - Y[base_k,c])   [R,K,C]
 *   i = rows[r] (rows NULL: i = r). hop_off == NULL: a dense row block, hop row i at hop + i*ld_hop with ncols = N columns (B = 1);
 *   else packed graphs as in gnan_aggregate_blockdiag_fwd, i a global node id, ncols >= the largest graph. T (table_per_row) and
 *   rscale rows are indexed by i; every i must be a row of the block / a node of the batch (not checked on the device). Any C;
 *   GNAN_ERR_UNSUPPORTED when one hop row with its weights and histogram does not fit shared memory. B >= 1 here, B >= 0 for
 *   the segment table and the graph rows (no graphs: nothing to do).
 * Work is rows x exceptions, each output element is a fixed-order sum written once (deterministic, no workspace). */
int gnan_explain_segments(const int64_t *grp_ptr /* [K+1] */, const int64_t *ent_row /* [E] */, int32_t K, const int32_t *node_off /* [B+1] */,
                          int32_t B, int64_t *seg /* [K,B+1] */, gnan_stream_t stream);
int gnan_explain_graph_features(const float *Y, const int64_t *grp_ptr, const int64_t *ent_row, const int64_t *seg, int32_t K, int32_t B,
                                int32_t C, const float *colw /* [N,C] */, const float *colw_sum /* [B,C] */, float *F /* [B,K,C] */,
                                gnan_stream_t stream);
int gnan_explain_rows_features(const uint8_t *hop, int64_t ld_hop, const int64_t *hop_off /* [B+1] or NULL */, const int32_t *node_off,
                               int32_t B, int64_t ncols, const int64_t *rows /* [R] or NULL */, int64_t R, const float *T, int table_per_row,
                               int32_t nbins, int32_t Cr, const float *rscale /* or NULL */, const float *Y, const int64_t *grp_ptr,
                               const int64_t *ent_row, const int64_t *seg, int32_t K, int32_t C, float *F /* [R,K,C] */,
                               gnan_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * The tail of the training step (csrc/train.cu; replaces trainer.py:52-67 and torch.optim.Adam.step, main.py:141).
 * Losses: *loss (device float, overwritten) = scale * sum of the per-sample terms (scale = 1/M for the reference's mean
 * reduction) and, when dlogits != NULL, d(loss)/d(logits) for an upstream gradient of 1 in the same pass.
 *   cross_entropy_rows: samples are the rows rows[m] (NULL: row m) of logits [N,C] with class labels[m]; dlogits is the FULL
 *     [N,C] gradient, zero on the rows without a loss (what the aggregation backward skips). An index outside [0,N) / label
 *     outside [0,C) sets *bad_index_flag (device int32, zero-initialised by the caller) and that sample is ignored.
 *   bce_with_logits: torch.nn.BCEWithLogitsLoss on logits [M], targets [M] in [0,1].
 * workspace: gnan_loss_workspace_bytes(). Deterministic (fixed summation order; unique rows).
 * adam_step: torch.optim.Adam semantics (no amsgrad, L2 weight_decay added to the gradient) for n_tensors fp32 tensors in one
 * launch: HOST arrays of device pointers / element counts; state = 3 device floats {step, 1-beta1^step, sqrt(1-beta2^step)},
 * zero-initialised by the caller and advanced by the call (so a captured CUDA graph keeps counting).
 * ---------------------------------------------------------------------------------------------- */
size_t gnan_loss_workspace_bytes(void);
int gnan_cross_entropy_rows(const float *logits, int64_t N, int32_t C, const int64_t *rows /* [M] or NULL */, const int64_t *labels,
                            int64_t M, float scale, float *loss, float *dlogits /* [N,C] or NULL */, int32_t *bad_index_flag,
                            void *workspace, size_t workspace_bytes, gnan_stream_t stream);
int gnan_bce_with_logits(const float *logits, const float *targets, int64_t M, float scale, float *loss, float *dlogits /* [M] or NULL */,
                         void *workspace, size_t workspace_bytes, gnan_stream_t stream);
int gnan_adam_step(int32_t n_tensors, float *const *params, const float *const *grads, float *const *exp_avg, float *const *exp_avg_sq,
                   const int64_t *numel, float *state /* [3] device */, float lr, float beta1, float beta2, float eps, float weight_decay,
                   gnan_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * All-pairs hop distances (replaces scipy dijkstra + the per-element normaliser loop,
 * pre_process_datasets.py:109-121,128-140; networkx BFS of batched_pyg_main.py:36-44).
 * Directed CSR (edges followed src -> dst), simple graph, unit weights. hop bytes: level, 255 = unreachable;
 * a finite level > 254 sets *overflow_flag (device int32) != 0.
 * cnt[i,d] = #{j: hop[i,j] = d} for d < nbins-1, cnt[i,nbins-1] = #unreachable; levels >= nbins-1 also set the flag.
 * ---------------------------------------------------------------------------------------------- */
/* Directed CSR (rowptr [N+1], col [E]) of the edge list src -> dst, built on the device by a counting sort on the source
 * (replaces the COO -> LIL conversion of pre_process_datasets.py:109,129). Neighbour order inside a row is unspecified.
 * *status (device int32): bit 0 = an endpoint outside [0,N) (that edge is dropped), bit 1 = duplicate (src,dst) pairs exist
 * (the reference sums them into weight-2 edges; the caller must subdivide them, see gnan_b200/preprocess.py). */
size_t gnan_build_csr_workspace_bytes(int32_t N, int64_t E);
int gnan_build_csr(const int64_t *src, const int64_t *dst, int64_t E, int32_t N, int32_t *rowptr, int32_t *col, int32_t *status,
                   void *workspace, size_t workspace_bytes, gnan_stream_t stream);

/* Edge list of a batch of B small graphs (<= 256 nodes each) from its compact TRANSFER form: src / dst [E] are uint8 node indices
 * INSIDE the edge's graph, edge_off [B+1] (int32) the first edge of each graph (edges grouped by graph), node_off [B+1] the graph
 * boundaries in the concatenated node set. Writes the PyG edge_index int64 [2,E] with global node ids (what gnan_build_csr
 * takes): 2 bytes per directed edge cross PCIe instead of 16 (batched_pyg_main.py:54-91 loader output). */
int gnan_edges_from_local(const uint8_t *src, const uint8_t *dst, const int32_t *edge_off, const int32_t *node_off, int32_t B,
                          int64_t E, int64_t *edge_index, gnan_stream_t stream);
/* The same with int16 endpoints (graphs of up to GNAN_APSP_BATCHED_MAX_NODES nodes; 4 bytes per directed edge). */
int gnan_edges_from_local_i16(const int16_t *src, const int16_t *dst, const int32_t *edge_off, const int32_t *node_off, int32_t B,
                              int64_t E, int64_t *edge_index, gnan_stream_t stream);

size_t gnan_apsp_bfs_workspace_bytes(int32_t N, int32_t n_sources);

/* sources [src_begin, src_end) of one graph with N nodes -> hop rows [src_end-src_begin, N] (row stride ld_hop). */
int gnan_apsp_bfs(const int32_t *rowptr /* [N+1] */, const int32_t *col /* [E] */, int32_t N, int32_t src_begin,
                  int32_t src_end, uint8_t *hop, int64_t ld_hop, int32_t *cnt /* [rows,nbins] or NULL */,
                  int32_t nbins, int32_t *overflow_flag, void *workspace, size_t workspace_bytes, gnan_stream_t stream);

/* Same result for a LARGE graph with a bit-parallel multi-source BFS (1024 sources per batch, one launch per level, pull
 * over out-neighbours so that every vertex writes its own row segment). Rows [row_begin,row_end), all N columns.
 * Exception to the "nothing synchronises" rule: the level count is data dependent, the stream is synchronised once per
 * group of 4 levels. cnt (if given) is zeroed by the callee. */
size_t gnan_apsp_msbfs_workspace_bytes(int32_t N);
int gnan_apsp_msbfs(const int32_t *rowptr, const int32_t *col, int32_t N, int32_t row_begin, int32_t row_end, uint8_t *hop,
                    int64_t ld_hop, int32_t *cnt, int32_t nbins, int32_t *overflow_flag, void *workspace,
                    size_t workspace_bytes, gnan_stream_t stream);

/* B graphs in one launch; CSR over the concatenated node set with GLOBAL column ids. max_n = the largest graph (sizes shared
 * memory; 1..GNAN_APSP_BATCHED_MAX_NODES); max_level (optional, zero-initialised by the caller) receives the largest finite hop of
 * the batch (atomicMax), which sizes the trimmed level table. order_ws is required scratch: [4*B+4] words, [5*B+5] when
 * max_n > 128.
 * Each graph runs by its own size:
 *  - at most 128 nodes: the graphs are grouped by size class, and a GROUP OF 4 WARPS works on one graph of 65..128 nodes, two of
 *    33..64 or four of up to 32 nodes at a time (one vertex per lane, a named barrier with an OR reduction per BFS level);
 *  - 129..GNAN_APSP_BATCHED_MAX_NODES nodes: one CTA per graph (one or two vertices per thread, 128 sources at a time).
 * Both launches go on `stream`, no synchronisation. max_n outside 1..GNAN_APSP_BATCHED_MAX_NODES: GNAN_ERR_UNSUPPORTED before any
 * CUDA call (gnan_apsp_bfs takes one graph of any size).
 * rscale (optional) [sumN,nbins] fp32 = 1/count (0 for an empty level), i.e. what gnan_level_rscale computes from cnt
 * (models.py:368-370 divides by the level size); cnt may then be NULL. Bit-identical to gnan_level_rscale of cnt at every graph
 * size: above 128 nodes the counts are summed across source chunks in the rscale rows (exact integers in fp32) and inverted once. */
int gnan_apsp_bfs_batched_ex(const int32_t *rowptr /* [sumN+1] */, const int32_t *col, const int32_t *node_off /* [B+1] */,
                             const int64_t *hop_off /* [B+1] */, int32_t B, int32_t max_n, uint8_t *hop,
                             int32_t *cnt /* [sumN,nbins] or NULL */, float *rscale, int32_t nbins, int32_t *overflow_flag,
                             int32_t *max_level, int32_t *order_ws /* [4*B+4], [5*B+5] if max_n > 128 */, gnan_stream_t stream);

/* gnan_apsp_bfs_batched_ex WITHOUT a CSR: the batch's edges in their transfer form (gnan_edges_from_local: src / dst uint8 indices
 * inside the graph, edge_off [B+1], edges grouped by graph). Every 4-warp group builds its graph's adjacency bit matrix in shared
 * memory from the graph's own edge segment; gnan_build_csr (and its ~0.1 ms per 4 M edges) drops out of a training step that
 * preprocesses its batch. Graphs of at most 128 nodes; order_ws [4*B+4] is required. *status (device int32, zeroed here) gets
 * gnan_build_csr's bits: 1 = an endpoint >= the graph's node count (edge dropped), 2 = a repeated (src,dst) pair (the reference
 * sums those into weight-2 edges: the caller must take the multi-edge path). pre_process_datasets.py:106-122 per graph. */
int gnan_apsp_bfs_batched_local(const uint8_t *src, const uint8_t *dst, const int32_t *edge_off, const int32_t *node_off,
                                const int64_t *hop_off, int32_t B, int32_t max_n, uint8_t *hop, int32_t *cnt, float *rscale,
                                int32_t nbins, int32_t *status, int32_t *overflow_flag, int32_t *max_level, int32_t *order_ws,
                                gnan_stream_t stream);

/* gnan_apsp_bfs_batched_local fused with gnan_aggregate_blockdiag_graph_fwd on the output-normaliser table (models.py:366-384 with
 * normalize_rho, a global table T [nbins,Cr]): the same out [B,C], colw [sumN,Cr] and Q [B,nbins,C] (gnan_aggregate_blockdiag_graph_bwd
 * is the backward), computed inside the BFS level loop. No hop bytes, level table or pair statistics are written. Directed graphs
 * are exact too. Same envelope as gnan_aggregate_blockdiag_graph_supported; *status (zeroed here), *overflow_flag and *max_level
 * (optional) as gnan_apsp_bfs_batched_local. Deterministic (fixed summation orders). Each graph runs by its own size:
 *  - at most 128 nodes: 4-warp groups as gnan_apsp_bfs_batched_local (a slower per-graph path for directed graphs);
 *  - 129..max_n nodes: one CTA per graph, 128 sources at a time, pulling over in-neighbours (exact for directed graphs in one pass);
 *    the in-neighbour bit matrix lives in shared memory (max_n^2 / 8 bytes), so no graph is refused for its edge count.
 * uint8 endpoints: max_n 1..256; order_ws [4*B+4] words, [5*B+5] when max_n > 128. A max_n outside the range is refused with
 * GNAN_ERR_UNSUPPORTED before any CUDA call. */
int gnan_bfs_graph_readout_fwd(const uint8_t *src, const uint8_t *dst, const int32_t *edge_off, const int32_t *node_off, int32_t B,
                               int32_t max_n, int32_t nbins, const float *T, int32_t Cr, const float *S, int32_t C, float *out,
                               float *colw, float *Q, int32_t *status, int32_t *overflow_flag, int32_t *max_level,
                               int32_t *order_ws /* [4*B+4], [5*B+5] if max_n > 128 */, gnan_stream_t stream);
/* The same with int16 endpoints (gnan_edges_from_local_i16's transfer form): max_n 1..GNAN_APSP_BATCHED_MAX_NODES. On the same
 * batch the results are bit-identical to gnan_bfs_graph_readout_fwd's. */
int gnan_bfs_graph_readout_fwd_i16(const int16_t *src, const int16_t *dst, const int32_t *edge_off, const int32_t *node_off, int32_t B,
                                   int32_t max_n, int32_t nbins, const float *T, int32_t Cr, const float *S, int32_t C, float *out,
                                   float *colw, float *Q, int32_t *status, int32_t *overflow_flag, int32_t *max_level,
                                   int32_t *order_ws /* [4*B+4], [5*B+5] if max_n > 128 */, gnan_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Deep graphs (csrc/wide.cu): hop distances > 254. The reference has no depth limit (pre_process_datasets.py:109-121), so the
 * same path exists with an int16 hop matrix (-1 = unreachable, levels 0..32766): warp-per-source BFS (no level table: the depth
 * is not known in advance; *max_level, zero-initialised by the caller, receives it and gnan_level_counts16 then builds the
 * [R, nbins] histogram, last column = unreachable), and the aggregation in its direct form (table lookups per pair, float atomics
 * for dT: not bit-reproducible). Slower than the uint8 kernels by design: taken only when the uint8 BFS reports an overflow.
 * ---------------------------------------------------------------------------------------------- */
size_t gnan_apsp_bfs16_workspace_bytes(int32_t N, int32_t n_sources);
int gnan_apsp_bfs16(const int32_t *rowptr, const int32_t *col, int32_t N, int32_t src_begin, int32_t src_end, int16_t *hop,
                    int64_t ld_hop, int32_t *overflow_flag, int32_t *max_level, void *workspace, size_t workspace_bytes,
                    gnan_stream_t stream);
int gnan_level_counts16(const int16_t *hop, int64_t R, int64_t N, int64_t ld_hop, int32_t *cnt, int32_t nbins, gnan_stream_t stream);
int gnan_aggregate_rows16_fwd(const int16_t *hop, int64_t R, int64_t N, int64_t ld_hop, const float *T, int table_per_row,
                              int32_t nbins, int32_t Cr, const float *rscale, const float *S, int32_t C, float *out,
                              gnan_stream_t stream);
int gnan_aggregate_rows16_bwd(const int16_t *hop, int64_t R, int64_t N, int64_t ld_hop, const float *T, int table_per_row,
                              int32_t nbins, int32_t Cr, const float *rscale, const float *S, int32_t C, const float *g, float *dS,
                              float *dT, uint8_t *row_flags_ws /* [R] scratch */, gnan_stream_t stream);

/* reference-format converters (pre_process_datasets.py:112-121): fp32 node_distances / normalization_matrix <-> hops */
int gnan_hops_to_reference(const uint8_t *hop, int64_t R, int64_t N, int64_t ld_hop, const int32_t *cnt, int32_t nbins,
                           float *node_distances, float *normalization_matrix, gnan_stream_t stream);
int gnan_hops_from_reference(const float *node_distances, const float *normalization_matrix /* or NULL */, int64_t R,
                             int64_t N, uint8_t *hop, int64_t ld_hop, int32_t *cnt /* or NULL; zero-initialised by caller */,
                             int32_t nbins, int32_t *overflow_flag, gnan_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GNAN_B200_H */
