/*
 * libmobgt — C-ABI of the B200-native (sm_100a) MobGT hot path.
 *
 * This is the drop-in boundary.  The reference (Yukayo/MobGT) has no C plugin
 * API: its hot path sits behind Python call sites.  Every entry point below
 * names the reference interface it replaces (file:line under
 * /root/reference/graphormer/).  Host code (mobgt_b200/*.py) binds these with
 * ctypes; see INTEGRATION.md for the stub a reference maintainer would add.
 *
 * Conventions
 *   - every function returns int32 status: 0 = OK, <0 = MOBGT_ERR_*; never throws
 *   - mobgt_last_error() returns a thread-local message for the last failure
 *   - pointers are DEVICE pointers unless the name ends in _host
 *   - no ownership transfer: the caller allocates inputs, outputs and workspaces
 *   - kernels are enqueued on `stream` (a cudaStream_t passed as void*) and the
 *     call never synchronises, so every call is CUDA-graph capturable
 *   - there is no CPU fallback anywhere in this library
 */
#ifndef MOBGT_H_
#define MOBGT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MOBGT_OK 0
#define MOBGT_ERR_BAD_SHAPE (-1)
#define MOBGT_ERR_BAD_DTYPE (-2)
#define MOBGT_ERR_UNSUPPORTED (-3)
#define MOBGT_ERR_CUDA (-4)
#define MOBGT_ERR_WORKSPACE_TOO_SMALL (-5)
#define MOBGT_ERR_NULL (-6)

#define MOBGT_UNREACHABLE 510 /* algos.pyx:32 — the reference's "infinity" */
#define MOBGT_MAX_NODES 512   /* rel_pos_encoder has 512 rows (model_fqandtoyo.py:788); the collator's default cap */
#define MOBGT_MAX_APSP_NODES 1024 /* K1 alone (the algos drop-in): graphs the model cannot take still get M, path, edges */
#define MOBGT_MAX_MODEL_NODES 1024 /* K2 / K3: graphs of up to 1024 nodes, T <= 1025 tokens (the collator's large_graphs mode) */
#define MOBGT_MAX_HOPS 32

/* dtype tags for float tensors crossing the ABI */
#define MOBGT_F32 0
#define MOBGT_BF16 1

int32_t mobgt_version(void);
/* Copies the calling thread's last error message (NUL-terminated) into buf. */
int32_t mobgt_last_error(char *buf, size_t buflen);
/* Process-wide count of libmobgt kernel launches so far (bench.py reports the per-step delta). */
int32_t mobgt_launch_count(int64_t *out);
/* 0 if a CUDA device of compute capability 10.x is current, else MOBGT_ERR_CUDA. */
int32_t mobgt_device_check(void);

/* ------------------------------------------------------------------------------------------
 * K1 — preprocessing: batched all-pairs shortest paths + path-edge extraction.
 * Replaces algos.floyd_warshall (algos.pyx:9-54), algos.get_all_edges (:57-62) and
 * algos.gen_edge_input (:65-96) as driven by preprocess_item (wrapper.py:42-61,99) and
 * the hop-axis slice of the collators (collator.py:323).
 *
 * Graphs are packed: graph g has n[g] nodes (1..MOBGT_MAX_APSP_NODES = 1024) and owns n[g]^2
 * cells starting at cell offset sq_off[g] of every per-cell array.  The model's kernels (K2/K3)
 * take at most MOBGT_MAX_NODES = 512; larger graphs are for the algos drop-in.
 *   feat      u8  [sum n^2]       attn_edge_type (wrapper.py:49-53): 0 = no edge, else
 *                                 edge feature (count+2).  adjacency = (feat != 0).
 *   dist      i16 [sum n^2]       M + shift        (M in 0..509 | 510)          (out)
 *   path      i16 [sum n^2]       FW `path` matrix (0..n-1 | 510), may be NULL  (out)
 *   edge_in   u8  [sum n^2, hops] e + shift; "no hop" (-1 in the reference) is stored
 *                                 as (uint8)(-1 + shift): 255 raw / 0 shifted   (out)
 *   maxdist   i32 [G]             max(M) per graph (wrapper.py:58)              (out)
 * shift = 0 gives the raw algos.pyx values, shift = 1 the collated ones
 * (pad_rel_pos_unsqueeze / pad_3d_unsqueeze "+1", collator.py:76-93).
 * hops = bytes per edge_in row (a multiple of 4, <= 32); dk = multi_hop_max_dist, the hop slots actually
 * walked (1 <= dk <= hops; the reference's default is 5, entry.py / data.py:204): slots [dk, hops) stay "no hop".
 * gids (i32 [G_launch], may be NULL = identity) selects which graphs this launch covers;
 * n_max_host is the largest n among them (chooses the cluster size / shared-memory plan).
 * n_max_host > 1024 returns MOBGT_ERR_BAD_SHAPE.  n_max_host > 512 needs a non-null `path`
 * (else MOBGT_ERR_NULL): that plan keeps only M in shared memory, writes `path` to global memory
 * and expands it into edge_in with a second kernel of the same call; MOBGT_ERR_UNSUPPORTED if its
 * cluster (8 or 16 CTAs) cannot be resident on the device.
 * ------------------------------------------------------------------------------------------ */
int32_t mobgt_apsp_edge_input(const uint8_t *feat, const int32_t *n, const int64_t *sq_off,
                              const int32_t *gids, int32_t G_launch, int32_t n_max_host,
                              int32_t hops, int32_t dk, int32_t shift,
                              int16_t *dist, int16_t *path, uint8_t *edge_in, int32_t *maxdist,
                              void *stream);

/* Stand-alone mirror of algos.gen_edge_input(max_dist, path, edge_feat) (algos.pyx:65-96) for a
 * caller that already holds a floyd_warshall `path` matrix (i16, packed like above).
 * Writes the first `hops` hop slots (1..510); same encoding as edge_in above.  n_max_host <= 1024. */
int32_t mobgt_gen_edge_input(const int16_t *path, const uint8_t *feat, const int32_t *n,
                             const int64_t *sq_off, int32_t G, int32_t n_max_host, int32_t hops,
                             int32_t shift, uint8_t *edge_in, void *stream);

/* in_degree / out_degree exactly as wrapper.py:97-98 names them (row sums / column sums of the
 * bool adjacency), + shift, for packed nodes: node_off[g] = sum_{g'<g} n[g'].  i16 out. */
int32_t mobgt_degrees(const uint8_t *feat, const int32_t *n, const int64_t *sq_off,
                      const int64_t *node_off, int32_t G, int32_t shift,
                      int16_t *in_degree, int16_t *out_degree, void *stream);

/* poi_pos (collator.py:428-437): distance bin 1..num_bins-1 between the POIs of every ordered node pair, from a
 * device-resident [P,2] coordinate table (stand-in for the reference's P x P distance pickle + np.digitize).
 * x i32 [sum n] = 1-based POI id per packed node; poi_pos i16 [sum n^2]. */
int32_t mobgt_poi_pos(const int32_t *x, const int32_t *n, const int64_t *sq_off, const int64_t *node_off,
                      const float *latlon, float dist_max, int32_t num_bins, int32_t G, int32_t n_max_host,
                      int16_t *poi_pos, void *stream);

/* ------------------------------------------------------------------------------------------
 * K2 — attention-bias build.  Replaces model_fqandtoyo.py:1143-1216 (fp32 statement model.py:126-190).
 * Packed index inputs as written by K1 with shift = 1 (rel_pos = M+1, edge_in = e+1) plus
 * poi_pos (collator.py:428-437), all per ordered node pair of each graph.
 *   bias [B,H,T,Tp] (f32 or bf16; Tp = row pitch, multiple of 8): only rows/cols < n[g]+1 are written;
 *   padding columns are masked inside the attention kernel from the sequence lengths.
 *   H = num_heads: built for 8 and 12; any other value returns MOBGT_ERR_UNSUPPORTED.
 *   tables: R [512,H] rel_pos_encoder, Ppos [bins,H] poi_pos_encoder, E [128,H] edge_encoder,
 *           W [>=hops*H*H] edge_dis_encoder (viewed [k,h',h]), tvd [H] graph_token_virtual_distance.
 *   hops is the byte stride of an edge_in row (a multiple of 4, as written by K1); dk = multi_hop_max_dist is the number of
 *   live hop slots and the clamp of the mean (sp = clamp(M, 1, dk), model_fqandtoyo.py:1168-1174); 1 <= dk <= hops.
 *   forward workspace: mobgt_bias_fwd_workspace_bytes() (the E.W table [hops,128,H] and the rel_pos-keyed table RL [512,H]);
 *   backward workspace: mobgt_bias_bwd_heads_workspace_bytes(T, hops, num_bins, H) (mobgt_bias_bwd_workspace_bytes() is the
 *   same for H = 8).
 * Input domain (not checked on the device; K1 writes only values inside it):
 *   rel_pos in 0..511 (511: unreachable pair); poi_pos in 0..num_bins-1; edge_in bytes in 0..127, bytes [dk, hops) of
 *   every row 0; E row 0 (edge_encoder's padding row) zero.  Cells with rel_pos - 1 >= rel_pos_max are -inf in the forward.
 *   The backward never reads a dBias cell outside a graph's live (n[g]+1)^2 square, in row 0, or masked by rel_pos_max.
 * Backward: dBias -> dR [512,H], dPpos [bins,H], dE [128,H], dW [hops*H*H], dtvd [H]  (all overwritten).
 *   dbias_dtype MOBGT_F32:  one f32 [B,H,T,Tp] buffer holding the sum over layers (n_layers = 1);
 *   dbias_dtype MOBGT_BF16: n_layers bf16 [B,H,T,Tp] planes, layer_stride elements apart (mobgt_attn_bwd mode 2),
 *                           summed in fp32 inside the kernel.
 *   The result is bitwise reproducible (fixed-order histogram reductions; the rare path — walk bytes that deviate from the
 *   expected walk — accumulates in 64-bit fixed point, where the order of the atomics is immaterial).  `workspace` must be
 *   16-byte aligned.
 * ------------------------------------------------------------------------------------------ */
/* bytes of `workspace` mobgt_bias_fwd needs; < 0 on bad arguments */
int64_t mobgt_bias_fwd_workspace_bytes(int32_t hops, int32_t H);
int32_t mobgt_bias_fwd(const int32_t *n, const int64_t *sq_off, const int16_t *rel_pos, const int16_t *poi_pos,
                       const uint8_t *edge_in, int32_t B, int32_t T, int32_t Tp, int32_t hops, int32_t dk, int32_t H,
                       int32_t rel_pos_max, int32_t num_bins, const float *R, const float *Ppos, const float *E,
                       const float *W, const float *tvd, void *workspace, void *out, int32_t out_dtype, void *stream);
/* bytes of `workspace` mobgt_bias_bwd needs at 8 heads (per-CTA partial histograms + totals); < 0 on bad arguments */
int64_t mobgt_bias_bwd_workspace_bytes(int32_t T, int32_t hops, int32_t num_bins);
/* the same at H heads (8 or 12); < 0 on bad arguments or another head count */
int64_t mobgt_bias_bwd_heads_workspace_bytes(int32_t T, int32_t hops, int32_t num_bins, int32_t H);
int32_t mobgt_bias_bwd(const int32_t *n, const int64_t *sq_off, const int16_t *rel_pos, const int16_t *poi_pos,
                       const uint8_t *edge_in, int32_t B, int32_t T, int32_t Tp, int32_t hops, int32_t dk, int32_t H,
                       int32_t rel_pos_max, int32_t num_bins, const void *dBias, int32_t dbias_dtype, int32_t n_layers,
                       int64_t layer_stride, const float *E, const float *W, void *workspace, int64_t workspace_bytes,
                       float *dR, float *dPpos, float *dE, float *dW, float *dtvd, void *stream);

/* K2, direct edge encoding (Graphormer's encoding for any edge_type other than multi_hop): the edge term of a pair is
 * E[f][h] with f = attn_edge_type of the pair, instead of the walk mean through edge_dis_encoder.
 *   bias[g,h,a,b] = R[rel_pos][h] + Ppos[poi_pos][h] + E[feat][h]   (a, b >= 1; indices of pair (a-1, b-1));
 *   column 0 of rows 1..n[g] = tvd[h]; row 0 = 0; -inf where rel_pos - 1 >= rel_pos_max; same [B,H,T,Tp] layout and
 *   written cells as mobgt_bias_fwd.  H = 8 or 12; any other value returns MOBGT_ERR_UNSUPPORTED.
 *   feat: packed u8 [sum n^2] (the batch's feat8 plane: 0 for no edge, else edge count + 2).
 * Input domain (not checked on the device): feat in 0..127; rel_pos in 0..511; poi_pos in 0..num_bins-1.  E row 0 is read
 *   for pairs without an edge (it need not be zero).
 * Backward: dBias (one f32 buffer or n_layers bf16 planes layer_stride elements apart, as mobgt_bias_bwd) -> dR [512,H],
 *   dPpos [bins,H], dE [128,H], dtvd [H] (all overwritten).  dE row 0 (edge_encoder's padding row) is 0: only pairs with
 *   feat != 0 contribute to dE.  There is no edge_dis_encoder gradient.  The backward never reads a dBias cell outside a
 *   graph's live (n[g]+1)^2 square, in row 0, or masked by rel_pos_max.  Bitwise reproducible (fixed-order histogram sums;
 *   dE and rel_pos keys outside the histogram plan accumulate in 64-bit fixed point).  `workspace` must be 16-byte aligned. */
int32_t mobgt_bias_direct_fwd(const int32_t *n, const int64_t *sq_off, const int16_t *rel_pos, const int16_t *poi_pos,
                              const uint8_t *feat, int32_t B, int32_t T, int32_t Tp, int32_t H, int32_t rel_pos_max,
                              int32_t num_bins, const float *R, const float *Ppos, const float *E, const float *tvd, void *out,
                              int32_t out_dtype, void *stream);
/* bytes of `workspace` mobgt_bias_direct_bwd needs; < 0 on bad arguments or a head count other than 8 and 12 */
int64_t mobgt_bias_direct_bwd_workspace_bytes(int32_t T, int32_t num_bins, int32_t H);
int32_t mobgt_bias_direct_bwd(const int32_t *n, const int64_t *sq_off, const int16_t *rel_pos, const int16_t *poi_pos,
                              const uint8_t *feat, int32_t B, int32_t T, int32_t Tp, int32_t H, int32_t rel_pos_max,
                              int32_t num_bins, const void *dBias, int32_t dbias_dtype, int32_t n_layers, int64_t layer_stride,
                              void *workspace, int64_t workspace_bytes, float *dR, float *dPpos, float *dE, float *dtvd,
                              void *stream);

/* ------------------------------------------------------------------------------------------
 * K3 — biased multi-head attention (tcgen05 / TMEM / TMA).  Replaces the core of
 * MultiHeadAttention.forward, model_fqandtoyo.py:1693-1706, for packed var-len graphs:
 * graph g owns token rows tok_off[g]..tok_off[g+1] (row 0 = graph token).  d = the head dim: 24 for the entry points
 * without a head_dim argument; the _hd variants take it as head_dim, built for 16 and 24 (any other value returns
 * MOBGT_ERR_UNSUPPORTED).
 *   q,k,v  bf16 [ntok, H*d] with a common row stride (elements) — usually slices of one fused projection
 *   bias   bf16 [B,H,T,Tp] from mobgt_bias_fwd ;  out bf16 [ntok, H*d] ;  lse f32 [ntok, H]
 *   drop_p, seed, seed_dev: the attention dropout of model_fqandtoyo.py:1704 (`x = self.att_dropout(x)` on the softmax
 *          probabilities; training only — pass drop_p = 0 in eval).  The keep mask is a counter-based hash of
 *          (seed, plane, row, column), regenerated by the backward from the SAME seed: nothing is stored.  seed_dev (u64 in
 *          device memory, optional) is folded into the seed at run time (CUDA-graph replays draw fresh masks).
 *   t_max_host / t_min_host: the largest / smallest token count (n + 1) of a graph of the batch, known on the host.  Graphs of
 *          at most 16 tokens (9 in 10 of a trajectory data set: median 4 nodes) are computed by a SIMT kernel (one 64-thread
 *          CTA per (graph, 4 heads), fp32 math, only the live bias cells are read), larger ones by the tensor-core kernel; both
 *          kernels select their graphs ON THE DEVICE from tok_off, the two host numbers only let the entry point skip a launch
 *          that would find no graph.  t_min_host = 0: unknown (both kernels are launched — e.g. when the call is captured
 *          in a CUDA graph that is replayed for other batches).
 *   graph_order: i32 [B] (optional) — the graph ids in launch order, largest graph first: CTA b works on graph
 *          graph_order[b / H], so the long-running CTAs start at once and the ones that find nothing to do are dispatched
 *          behind them.  NULL: identity.
 * ------------------------------------------------------------------------------------------ */
int32_t mobgt_attn_fwd(const void *q, const void *k, const void *v, int64_t qkv_row_stride, const void *bias,
                       const int32_t *tok_off, const int32_t *graph_order, int32_t B, int32_t H, int32_t ntok, int32_t T, int32_t Tp,
                       int32_t t_max_host, int32_t t_min_host, float scale, float drop_p, uint64_t seed, const void *seed_dev,
                       void *out, float *lse, void *stream);
int32_t mobgt_attn_fwd_hd(const void *q, const void *k, const void *v, int64_t qkv_row_stride, const void *bias,
                          const int32_t *tok_off, const int32_t *graph_order, int32_t B, int32_t H, int32_t ntok, int32_t T,
                          int32_t Tp, int32_t t_max_host, int32_t t_min_host, float scale, float drop_p, uint64_t seed,
                          const void *seed_dev, void *out, float *lse, int32_t head_dim, void *stream);

/* Backward of mobgt_attn_fwd.  o, dout: bf16 [ntok, H*d] contiguous; lse from the forward.
 * dq, dk, dv: bf16 with a common row stride (usually slices of one [ntok, 3*H*d] buffer).
 * dbias receives dS = d(scores) = d(bias) [B,H,T,Tp]:
 *   mode 0: f32, overwritten ;  mode 1: f32, added to (the bias is shared by all encoder layers) ;
 *   mode 2: bf16, overwritten by ONE TMA store per tile from the MMA operand image — each layer writes its own plane and
 *           mobgt_bias_bwd sums the planes in fp32 (no read-modify-write traffic; rows / columns past a graph's
 *           tokens receive unspecified values and are never read).
 * Scores / probabilities are recomputed in-tile and never stored in HBM. */
int32_t mobgt_attn_bwd(const void *q, const void *k, const void *v, int64_t qkv_row_stride, const void *bias,
                       const void *o, const void *dout, const float *lse, const int32_t *tok_off, const int32_t *graph_order,
                       int32_t B, int32_t H, int32_t ntok, int32_t T, int32_t Tp, int32_t t_max_host, int32_t t_min_host, float scale,
                       void *dq, void *dk, void *dv, int64_t dqkv_row_stride, void *dbias, int32_t mode, float drop_p,
                       uint64_t seed, const void *seed_dev, void *stream);
int32_t mobgt_attn_bwd_hd(const void *q, const void *k, const void *v, int64_t qkv_row_stride, const void *bias,
                          const void *o, const void *dout, const float *lse, const int32_t *tok_off, const int32_t *graph_order,
                          int32_t B, int32_t H, int32_t ntok, int32_t T, int32_t Tp, int32_t t_max_host, int32_t t_min_host,
                          float scale, void *dq, void *dk, void *dv, int64_t dqkv_row_stride, void *dbias, int32_t mode,
                          float drop_p, uint64_t seed, const void *seed_dev, int32_t head_dim, void *stream);

/* K3 in fp32 mode: the same attention core (model_fqandtoyo.py:1693-1706) with fp32 q / k / v / bias / out and fp32 math
 * (IEEE expf / logf, SIMT), for graphs of any size up to 513 tokens — the arithmetic of the reference's `--precision 32`
 * (Lightning's default).  It exists for the first half of the parity contract ("within 1e-5 relative in fp32 mode"): the
 * tensor-core kernels above round their operands to bf16 by construction.  Same packed layout, same dropout mask (seed, plane,
 * row, column) as mobgt_attn_fwd; lse is the natural-log row normaliser.  dbias f32 [B,H,T,Tp]: mode 0 overwritten, mode 1
 * added to (only the live cells of a graph are touched); feed it to mobgt_bias_bwd with dbias_dtype MOBGT_F32, n_layers 1.
 * Bitwise reproducible (fixed-order shuffle reductions, no atomics).  Head dim 24; the _hd variants take it as head_dim
 * (built: 16, 24; anything else returns MOBGT_ERR_UNSUPPORTED). */
int32_t mobgt_attn_f32_fwd(const float *q, const float *k, const float *v, int64_t qkv_row_stride, const float *bias,
                           const int32_t *tok_off, int32_t B, int32_t H, int32_t ntok, int32_t T, int32_t Tp, int32_t t_max_host,
                           float scale, float drop_p, uint64_t seed, const void *seed_dev, float *out, float *lse, void *stream);
int32_t mobgt_attn_f32_bwd(const float *q, const float *k, const float *v, int64_t qkv_row_stride, const float *bias,
                           const float *o, const float *dout, const float *lse, const int32_t *tok_off, int32_t B, int32_t H,
                           int32_t ntok, int32_t T, int32_t Tp, int32_t t_max_host, float scale, float *dq, float *dk, float *dv,
                           int64_t dqkv_row_stride, float *dbias, int32_t mode, float drop_p, uint64_t seed, const void *seed_dev,
                           void *stream);
int32_t mobgt_attn_f32_fwd_hd(const float *q, const float *k, const float *v, int64_t qkv_row_stride, const float *bias,
                              const int32_t *tok_off, int32_t B, int32_t H, int32_t ntok, int32_t T, int32_t Tp,
                              int32_t t_max_host, float scale, float drop_p, uint64_t seed, const void *seed_dev, float *out,
                              float *lse, int32_t head_dim, void *stream);
int32_t mobgt_attn_f32_bwd_hd(const float *q, const float *k, const float *v, int64_t qkv_row_stride, const float *bias,
                              const float *o, const float *dout, const float *lse, const int32_t *tok_off, int32_t B, int32_t H,
                              int32_t ntok, int32_t T, int32_t Tp, int32_t t_max_host, float scale, float *dq, float *dk, float *dv,
                              int64_t dqkv_row_stride, float *dbias, int32_t mode, float drop_p, uint64_t seed,
                              const void *seed_dev, int32_t head_dim, void *stream);

/* ------------------------------------------------------------------------------------------
 * K4 — node-embedding gather / sum and the deterministic segmented scatter-add backward.
 * Replaces model_fqandtoyo.py:1257-1269 (per-node table look-ups) and :1288-1344 (degree encoders,
 * positional rows, graph token).  Packed nodes / tokens, no padding rows.
 *   gather: out[v] = Gd[x[v]-1] | Tm[slot[v]] | Gc[cat_of_poi[x[v]-1]-1]   (widths Dp | Dt | Dc)
 *   sum:    tok[r] = pos==0 ? graph_token + pe[0] : nf[node] + Din[in_deg] + Dout[out_deg] + pe[pos]
 *   segment_sum: table[key] = sum of src rows with that key, in the order of a stable sort
 *                (perm, keys_sorted); no atomics -> bitwise reproducible.
 * ------------------------------------------------------------------------------------------ */
int32_t mobgt_embed_gather_fwd(const int32_t *x, const int32_t *slot, const int32_t *cat_of_poi, const float *Gd,
                               const float *Tm, const float *Gc, int32_t nnode, int32_t Dp, int32_t Dt, int32_t Dc,
                               void *out, int32_t out_dtype, void *stream);
int32_t mobgt_embed_sum_fwd(const void *nf, const int32_t *tok_graph, const int32_t *tok_pos, const int32_t *in_deg,
                            const int32_t *out_deg, const float *Din, const float *Dout, const float *pe,
                            const float *graph_token, int32_t ntok, int32_t D, void *tok, int32_t dtype, void *stream);
int32_t mobgt_segment_sum(const void *src, int32_t src_dtype, int64_t src_stride, int32_t col0, int32_t D,
                          const int32_t *perm, const int32_t *keys_sorted, int32_t nrows, float *table, int32_t nkeys,
                          void *workspace, int64_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------
 * K6 — encoder row ops next to the attention path (SURVEY.md §8f #2, first slice).  Replace nn.LayerNorm forward / backward
 * (EncoderLayer ffn_norm1 / ffn_norm2 and final_ln, model_fqandtoyo.py:1731-1743, :1360-1364; biased variance, eps inside the
 * sqrt) and the bias gradient dy.sum(0) of every nn.Linear on the path.
 *   layernorm_fwd: x f32 [N,D] -> out f32 [N,D] (+ optional bf16 copy for the next GEMM), mean / rstd f32 [N] for backward.
 *   layernorm_bwd: dy f32 and/or dy_bf16 [N,D] (summed when both are given) -> dx f32 [N,D], dgamma / dbeta f32 [D]
 *                  (deterministic two-stage reduction; workspace: mobgt_layernorm_bwd_workspace_bytes(D)).
 *   add_dropout_layernorm_fwd / _bwd: the post-LN residual block  s = x + dropout(y) ; out = LayerNorm(s)  in one pass
 *                  (x f32 residual stream, y bf16 sub-layer output; s_out f32 = the new residual stream, optional).  The mask
 *                  is a counter-based hash of (seed, element index), regenerated in backward: nothing is stored.  seed_dev
 *                  (u64 in device memory, optional) is folded into the seed at run time, so a CUDA graph that replays the
 *                  kernels with baked-in arguments draws a fresh mask per replay (increment it inside the graph).  Backward:
 *                  ds = LayerNorm-backward(dy [+ dy_bf16]) + ds_ext (gradient reaching s from its later uses, optional);
 *                  dx = ds ; dyb_out (bf16, optional) = ds * mask / (1 - p) ; dyb_colsum (f32 [D], optional) = the column sums of
 *                  dyb_out, i.e. the bias gradient of the nn.Linear whose output y was (no separate column-sum pass).
 *   colsum:        out[c] = sum_r src[r, c]  (src bf16 or f32, row stride in elements; fp32 accumulation, fixed order).
 *   D multiple of 32 with D/32 in {2,4,6,8,10,12,16}.
 * ------------------------------------------------------------------------------------------ */
int32_t mobgt_layernorm_fwd(const float *x, const float *gamma, const float *beta, float eps, int32_t N, int32_t D, float *out,
                            void *out_bf16, float *mean, float *rstd, void *stream);
int64_t mobgt_layernorm_bwd_workspace_bytes(int32_t D);
int32_t mobgt_layernorm_bwd(const float *dy, const void *dy_bf16, const float *x, const float *gamma, const float *mean,
                            const float *rstd, int32_t N, int32_t D, float *dx, float *dgamma, float *dbeta, void *workspace,
                            int64_t workspace_bytes, void *stream);
int32_t mobgt_add_dropout_layernorm_fwd(const float *x, const void *y_bf16, float drop_p, uint64_t seed, const float *gamma,
                                        const float *beta, float eps, int32_t N, int32_t D, float *s_out, float *out, void *out_bf16,
                                        float *mean, float *rstd, const void *seed_dev, void *stream);
int32_t mobgt_add_dropout_layernorm_bwd(const float *dy, const void *dy_bf16, const float *ds_ext, const float *s_saved,
                                        const float *gamma, const float *mean, const float *rstd, int32_t N, int32_t D, float drop_p,
                                        uint64_t seed, float *dx, void *dyb_out, float *dgamma, float *dbeta, float *dyb_colsum,
                                        void *workspace, int64_t workspace_bytes, const void *seed_dev, void *stream);
int64_t mobgt_colsum_workspace_bytes(int32_t N, int32_t C);
int32_t mobgt_colsum(const void *src, int32_t src_dtype, int64_t src_stride, int32_t N, int32_t C, float *out, void *workspace,
                     int64_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------
 * K5 — POI-logit head fused with per-row top-k and rank counting.  Replaces out_proj followed by get_acc / MRR_metric
 * (model_fqandtoyo.py:1396-1428, :48-90, :122-131).  logits = z W^T + bias are produced tile by tile in TMEM and
 * consumed in the epilogue; they are only written to HBM when logits_dump != NULL (tests).
 *   z bf16 [M,K] ; W bf16 [V,K] = this rank's vocabulary shard (global index of row 0 = vocab_offset) ; bias f32 [V]|NULL
 *   target i32 [M] global vocabulary index (<0: none) ; K multiple of 16, <= 320 ; k <= 32 ; nsplit even, <= 160
 *   mode 0: st[row] = logit of the row's target, written by the shard that owns it (initialise st to -inf; across
 *           shards: all-reduce MAX)
 *   mode 1: per (row, split): sorted top-k (value, global index), count(s > st), count(s == st and idx < target)
 *   thr_share: u32 [M] zero-initialised scratch or NULL.  Every list of a row publishes its k-th value there (atomic max of
 *           order-preserving bits); since the k-th value of ANY subset bounds the row's final k-th value from below, all
 *           lists of the row (all splits, and — over NVLink peer memory or after an all-reduce MAX — all shards) prune
 *           with it.  The merged top-k is unchanged; lists may come back shorter than k (index -1 = empty slot).
 * mobgt_topk_merge merges S sorted lists per row (ties -> lower index) and sums the counts into rank[M].
 * ------------------------------------------------------------------------------------------ */
int32_t mobgt_head_topk(const void *z, const void *W, const float *bias, const int32_t *target, int32_t M, int32_t V,
                        int32_t K, int64_t vocab_offset, int32_t k, int32_t nsplit, int32_t mode, float *st,
                        float *topk_val, int32_t *topk_idx, int32_t *cnt_gt, int32_t *cnt_eq, float *logits_dump,
                        void *thr_share, void *stream);
int32_t mobgt_topk_merge(const float *val, const int32_t *idx, const int32_t *cnt_gt, const int32_t *cnt_eq, int32_t M,
                         int32_t S, int32_t k, float *out_val, int32_t *out_idx, int32_t *rank, void *stream);

/* K5 in fp32 mode (`--precision 32` evaluation): the same head with z f32 [M,K] and W f32 [V,K] (out_proj.weight itself),
 * logits in IEEE fp32 on the CUDA cores (no tensor-core instruction).  Every logit is computed in ONE fixed order,
 *     s = 0;  for k = 0 .. K-1 ascending: s = fmaf(z[row][k], W[col][k], s);   logit = bias ? s + bias[col] : s
 * (each fmaf and the add rounded once), whatever the tiling, nsplit or vocabulary shard: results are bitwise reproducible.
 * mode 0 runs the same chain for the target's column, so the target's own logit equals st and never counts against itself.
 *   K multiple of 4, 4 <= K <= 320 ; 1 <= k <= 32 ; mode 1: nsplit = 4 x (vocabulary splits), a multiple of 4 in [4, 160]
 *   z and W 16-byte aligned (rows are then too, K being a multiple of 4); bias f32 [V] or NULL, any 4-byte alignment
 *   mode 1 outputs per (row, list), same layout and meaning as mobgt_head_topk: a sorted top-k (value, global index; ties ->
 *   lower index; a list may hold fewer than k entries: index -1), cnt_gt = #(s > st), cnt_eq = #(s == st and idx < target);
 *   mobgt_topk_merge gives rank = cnt_gt + cnt_eq.  logits_dump (optional [M,V] f32) receives the kernel's own logits.
 *   thr_share is not used (the lists of a row prune independently): pass NULL.
 * Bad arguments return MOBGT_ERR_NULL / MOBGT_ERR_BAD_SHAPE before any launch. */
int32_t mobgt_head_topk_f32(const float *z, const float *W, const float *bias, const int32_t *target, int32_t M, int32_t V,
                            int32_t K, int64_t vocab_offset, int32_t k, int32_t nsplit, int32_t mode, float *st,
                            float *topk_val, int32_t *topk_idx, int32_t *cnt_gt, int32_t *cnt_eq, float *logits_dump,
                            void *thr_share, void *stream);

/* ------------------------------------------------------------------------------------------
 * Test hooks (tests/test_umma_selftest.py): exercise the tcgen05 / TMA building blocks in isolation.
 * out[128,N] (f32) = A * B, bf16 operands; a_mn / b_mn select MN-major operands
 * (A: a_mn ? [K,128] : [128,K];  B: b_mn ? [K,N] : [N,K], all row-major).
 * ------------------------------------------------------------------------------------------ */
int32_t mobgt_selftest_umma(const void *A, const void *B, int32_t N, int32_t K, int32_t a_mn, int32_t b_mn,
                            float *out, void *stream);

/* Backward of the FFN's GELU (nn.GELU(), exact erf form; model_fqandtoyo.py:1650, applied :1654) on bf16 activations, fp32 math.
 *   gelu_bwd_colsum: dh = da * gelu'(h) (bf16 [N, C]) and dbias[c] = sum_r dh[r, c] (fp32, fixed order) — the input gradient of
 *                    the activation fused with the bias gradient of the Linear that produced h.  Workspace as mobgt_colsum. */
int32_t mobgt_gelu_bwd_colsum(const void *da_bf16, const void *h_bf16, int32_t N, int32_t C, void *dh_bf16, float *dbias,
                              void *workspace, int64_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------
 * K7 — training losses over the logits (SURVEY.md §8a A5b).  logits: f32 or bf16 [B, V] with row_stride elements between
 * rows; target: i64 [B] class ids.  Forward: ONE read of the logits; backward: one read + one write; `grad_out` is the
 * upstream gradient of the scalar loss in DEVICE memory (f32 [1]) so the call is CUDA-graph capturable.  Partials are merged
 * in a fixed order (bitwise reproducible).  workspace: mobgt_loss_workspace_bytes(B, V).
 *   lsm_nll: mean over the rows with target != ignore_index of -log_softmax(logits)[target]
 *            = log_softmax (model_fqandtoyo.py:1425) + NLLLoss(ignore_index=0) (data.py:165; model_fqandtoyo.py:1470-1471).
 *            lse f32 [B] (saved for backward), loss f32 [2] = {loss, number of live rows}.
 *   gtl:     GradientTailLoss(alpha, beta = 1, k = 1), model_fqandtoyo.py:545-550: mean over [B, V] of
 *            -alpha (1-p) log p on the target class and -p log(1-p) elsewhere, p = sigmoid(logit).  loss f32 [1].
 * dlogits has the dtype of logits.  Rows may be PADDED: row_stride >= V, and when d_row_stride exceeds V by fewer than 16 elements the
 * padding columns of dlogits are zero-filled (a head whose class count is padded to a multiple of 8 for the GEMMs: the padding
 * classes take no part in the loss and get no gradient).
 * ------------------------------------------------------------------------------------------ */
int64_t mobgt_loss_workspace_bytes(int32_t B, int32_t V);
int32_t mobgt_lsm_nll_fwd(const void *logits, int32_t dtype, int64_t row_stride, const int64_t *target,
                          int64_t ignore_index, int32_t B, int32_t V, void *workspace, int64_t workspace_bytes,
                          float *lse, float *loss, void *stream);
int32_t mobgt_lsm_nll_bwd(const void *logits, int32_t dtype, int64_t row_stride, const int64_t *target,
                          int64_t ignore_index, int32_t B, int32_t V, const float *lse, const float *loss,
                          const float *grad_out, void *dlogits, int64_t d_row_stride, void *stream);
int32_t mobgt_gtl_fwd(const void *logits, int32_t dtype, int64_t row_stride, const int64_t *target, float alpha,
                      int32_t B, int32_t V, void *workspace, int64_t workspace_bytes, float *loss, void *stream);
int32_t mobgt_gtl_bwd(const void *logits, int32_t dtype, int64_t row_stride, const int64_t *target, float alpha,
                      int32_t B, int32_t V, const float *grad_out, void *dlogits, int64_t d_row_stride, void *stream);

/* ------------------------------------------------------------------------------------------
 * K8 — CSR SpMM of the global GCN tables (SURVEY.md §8f #1).  Replaces torch.spmm(adj, support) of
 * GraphConvolution.forward (modelGNN.py:39-46; called for poi_distance_model / poi_cat_model every forward,
 * model_fqandtoyo.py:1236-1237):   Y[r,:] = act( sum_j val[j] * S[col[j],:] + bias ),  j over row r of the CSR matrix.
 *   crow i32 [nrows+1], col i32 [nnz], val f32 [nnz]; S f32 [ncols, D], Y f32 [nrows, D] contiguous; D in {16,32,64,128};
 *   bias f32 [D] or NULL; activation != 0: LeakyReLU(leaky_slope) (GCN.forward, modelGNN.py:67-69).
 * The backward w.r.t. S is the same call on the CSR of the transposed matrix (no atomics; bitwise reproducible).
 * ------------------------------------------------------------------------------------------ */
int32_t mobgt_spmm_csr(const int32_t *crow, const int32_t *col, const float *val, int32_t nrows, const float *S,
                       int32_t D, const float *bias, float leaky_slope, int32_t activation, float *Y, void *stream);

/* ------------------------------------------------------------------------------------------
 * K9 — AdamW over flat fp32 buffers (param, grad, exp_avg, exp_avg_sq: n elements each, n % 4 == 0, 16-byte aligned).
 * Replaces torch.optim.AdamW of configure_optimizers (model_fqandtoyo.py:1599-1616) in the training loop: one pass,
 * 28 B / parameter.  `step` is the 1-based update count (bias correction); decoupled weight decay, no amsgrad.
 * ------------------------------------------------------------------------------------------ */
int32_t mobgt_adamw_step(float *param, const float *grad, float *exp_avg, float *exp_avg_sq, int64_t n, float lr, float beta1,
                         float beta2, float eps, float weight_decay, int64_t step, void *stream);

/* ------------------------------------------------------------------------------------------
 * K10 — encoder GEMMs on tcgen05 / TMEM / TMA with fused epilogues (SURVEY.md §8f #2).  Replaces the nn.Linear calls of
 * the encoder layers and the element-wise kernels behind them (model_fqandtoyo.py:1644-1656, 1683-1685, 1708, 1731-1743).
 *   A bf16 [M, K] (row stride lda), B bf16 [N, K] (the nn.Linear weight layout, row stride ldb), bias f32 [N] or NULL,
 *   C bf16 [M, N] (row stride ldc).  N % 128 == 0, K % 16 == 0, strides % 8 == 0, 16-byte aligned pointers.
 *   mode 0: C = A B^T + bias ;  mode 1: C = gelu(A B^T + bias)  (nn.GELU(), exact erf form) ;
 *   mode 2: C = (A B^T) o gelu'(A2 B2^T + bias), A2 bf16 [M, K2], B2 bf16 [N, K2] — the FFN backward
 *           dh = (dy W2) o gelu'(x W1^T + b1) with the pre-activation recomputed; colsum f32 [N] (optional) = column sums
 *           of C, i.e. the bias gradient of layer1 (workspace: mobgt_gemm_workspace_bytes(M, N, 2)).
 * ------------------------------------------------------------------------------------------ */
int64_t mobgt_gemm_workspace_bytes(int32_t M, int32_t N, int32_t mode);
/* GELU of modes 1 / 2: 1 (default) = erf form (nn.GELU() to 1.5e-7); 0 = tanh form 0.5 x (1 + tanh(sqrt(2/pi) (x + 0.044715 x^3)))
 * on the hardware tanh unit, within 4.8e-4 absolute of the erf form and ~15 % faster — not the default because its derivative
 * error compounds over the layers (see csrc/k10_gemm.cu).  Forward and backward always use the same function.  Process-wide. */
int32_t mobgt_gemm_exact_gelu(int32_t on);
int32_t mobgt_gemm_bf16(const void *A, int64_t lda, const void *B, int64_t ldb, const float *bias, void *C, int64_t ldc,
                        int32_t M, int32_t N, int32_t K, int32_t mode, const void *A2, int64_t lda2, const void *B2,
                        int64_t ldb2, int32_t K2, float *colsum, void *workspace, int64_t workspace_bytes, void *stream);

/* Debug hook: register (NULL: clear) a device buffer of 256 int64; thread 0 of one CTA of mobgt_attn_fwd / mobgt_attn_bwd then
 * stamps clock64() at its pipeline stages (scripts/timeline.py). */
int32_t mobgt_debug_set_timeline(void *dev_buf256);
/* Measurement switch of mobgt_head_topk: 0 = never pair adjacent row tiles into 2-CTA clusters (TMA multicast of the W stages),
 * 1 = default (paired whenever the number of 128-row tiles is even). */
int32_t mobgt_debug_head_cluster(int32_t on);

#ifdef __cplusplus
}
#endif
#endif /* MOBGT_H_ */
