/*
 * edis.h -- C ABI of libedis.so: the B200 (sm_100a) DISGAT message-passing hot path.
 *
 * The reference (TianxiangZhao/EdgeDisentangle_SSL) is pure PyTorch and has no FFI; each
 * entry point below names the reference Python code it replaces (file:line under
 * /root/reference).  Conventions:
 *   - plain pointers and sizes only; no torch types.  All tensors fp32, row-major.
 *   - every `const float*` / `float*` argument of an op is a DEVICE pointer; the caller owns
 *     all of them (outputs and workspaces included).  The library allocates device memory
 *     only inside edis_graph_create and frees it in edis_graph_destroy.
 *   - ops are asynchronous on `stream` (a cudaStream_t passed as void*), stateless and
 *     re-entrant per stream.
 *   - return value 0 = ok, negative = error; edis_last_error() gives the message
 *     (thread-local).  There is no CPU fallback anywhere.
 *   - channel-fused layout: a "node tensor" is [N, C*D] with channel c in columns
 *     [c*D, (c+1)*D) (== torch.cat of the reference's per-channel [N, D] tensors, so
 *     FuseLayer's `torch.cat(feature_list, -1)`, layers.py:900, is free); an "edge tensor"
 *     is [E, C] in CSR (row-major, destination-sorted) edge order.
 */
#ifndef EDIS_H_
#define EDIS_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EDIS_OK 0
#define EDIS_ERR_ARG (-1)
#define EDIS_ERR_CUDA (-2)
#define EDIS_ERR_UNSUPPORTED (-3)
#define EDIS_ERR_WORKSPACE (-4)
#define EDIS_ERR_STALE (-5) /* edis_graph_load: cache file missing, corrupt, or written for other input */

const char* edis_last_error(void);
/* library / build identification: "edis <ver> sm_100a" */
const char* edis_version(void);

/* ------------------------------------------------------------------ graph builder (host)
 * Replaces data_load.py:39-77 (`load_data`: edge list / CSR -> dense N x N -> fill_diagonal ->
 * symmetrise by max -> row-normalise -> scipy CSR -> torch sparse COO) and utils.py:163-170
 * (`edge2adj`).  Integer work on HOST pointers, bit-exact structure and float32 values.
 *   rows/cols[m]  input entries (any order, duplicates allowed; duplicates keep the max value)
 *   vals[m]       entry values or NULL (= all 1)
 *   out_row/out_col/out_val  caller-allocated with capacity 2*m + n
 * Returns the number of entries E of the processed adjacency (row-major sorted), or <0. */
int64_t edis_build_adjacency_host(int64_t n, int64_t m, const int64_t* rows, const int64_t* cols,
                                  const double* vals, int64_t* out_row, int64_t* out_col,
                                  float* out_val);

/* ------------------------------------------------------------------ graph handle
 * Device-resident CSR (+ CSC for the source-side backward) of one adjacency, with the
 * chunked work schedules the kernels use.  Replaces the per-call `adj.coalesce().indices()`
 * of layers.py:344 (run 8x per DISGAT pass in the reference).
 *   row/col[e]  HOST pointers, COO of the adjacency.  If not already row-major sorted and
 *               duplicate-free it is sorted (stable) and `perm` reports the permutation.
 *   max_chunk   max edges one warp processes for one row (rows above are split); 0 = default
 * The CSR edge order equals the reference's coalesced order, so edge tensors line up with
 * the reference's `edge_e[k]` with no permutation.
 *   device      CUDA device ordinal, or -1 for a STRUCTURE-ONLY handle: host mirrors and schedules
 *               are built, nothing is uploaded; usable with edis_graph_info / edis_graph_export only
 *               (host-side checks of the builder) -- every op rejects it. */
typedef struct edis_graph edis_graph;
int edis_graph_create(int64_t n, int64_t e, const int64_t* row, const int64_t* col, int max_chunk,
                      int device, edis_graph** out);
/* Rectangular variant for a destination-range partition of a larger graph (multi-GPU): rows
 * are the n_rows destination nodes this rank owns, columns the n_cols >= n_rows source nodes it
 * reads (its own nodes FIRST, then halo nodes), so destination node i is also source node i.
 * Destination-side node tensors (out, hpre, g_out, gh, the P rows used) have n_rows rows,
 * source-side ones (Q, V, gQ, gV) n_cols rows. */
int edis_graph_create_rect(int64_t n_rows, int64_t n_cols, int64_t e, const int64_t* row,
                           const int64_t* col, int max_chunk, int device, edis_graph** out);
void edis_graph_destroy(edis_graph* g);

/* info[0]=n, [1]=e, [2]=dst items, [3]=dst partial slots, [4]=src items, [5]=src partial slots,
 * [6]=max in-degree, [7]=max out-degree, [8]=1 if the input was already sorted (perm = identity),
 * [9]=n_cols */
int edis_graph_info(const edis_graph* g, int64_t info[10]);
/* number of entries of the INPUT edge list the handle was built from (= length of `perm`) */
int64_t edis_graph_input_entries(const edis_graph* g);
/* copies of the structure arrays to HOST buffers (any may be NULL): rowptr[n+1], col[e],
 * perm[e_in] (input entry k -> CSR slot perm[k]; sized by the INPUT entry count, duplicates
 * map to the same slot), cscptr[n_cols+1], cscrow[e], csceid[e] */
int edis_graph_export(const edis_graph* g, int64_t* rowptr, int32_t* col, int64_t* perm,
                      int64_t* cscptr, int32_t* cscrow, int32_t* csceid);
/* bytes of scratch the layer ops need for a node tensor of `width` floats per row */
int64_t edis_graph_workspace_bytes(const edis_graph* g, int64_t width);

/* On-disk graph cache (SURVEY 8(f)3).  Replaces the per-start dense detour of data_load.py:39-77 /
 * utils.py:163-170 (39.5 s on cora_full) and, by construction, the stale-cache hazard of
 * pretrainer.py:390-398 (`./resource/<ds>/DisEdges.pt`, keyed by dataset name only): a file is
 * keyed by a 64-bit content key chosen by the caller and by max_chunk, and is rejected otherwise.
 *   edis_edge_list_key  content key of an input edge list (+ sizes and max_chunk): the key to use
 *                       when the cache stands for `edis_graph_create_rect` on exactly this input
 *   edis_graph_save     writes rowptr / col / perm / CSC / both schedules (+ heat bits) to `path`
 *                       atomically (temp file + rename)
 *   edis_graph_load     memory-maps `path`, checks magic / version / key / max_chunk / sizes (and the
 *                       payload checksum when verify != 0), uploads straight from the mapping to
 *                       `device` (-1: structure-only handle).  EDIS_ERR_STALE = no usable file (not
 *                       an error of the caller: rebuild and save). */
uint64_t edis_edge_list_key(int64_t n, int64_t n_cols, int64_t e_in, const int64_t* row,
                            const int64_t* col, int max_chunk);
int edis_graph_save(const edis_graph* g, const char* path, uint64_t key);
int edis_graph_load(const char* path, uint64_t key, int max_chunk, int device, int verify,
                    edis_graph** out);

/* ------------------------------------------------------------------ fused DisGALayer
 * One call computes ALL C channels of one DISGAT layer.  Replaces, per channel,
 * layers.py:349-416 (`DisGALayer.forward_sparse`: edge scoring -> sigmoid ->
 * utils.sp_softmax (utils.py:192-200) -> dropout -> utils.sp_matmul (utils.py:203-207)) and
 * the F.elu of layers.py:500/509.  The dense node projections stay torch GEMMs outside:
 *   att 1: sdst = (xW)a_top, ssrc = (xW)a_bot         -> P = sdst[N,C], Q = ssrc[N,C]
 *   att 2: h = xW                                     -> P = Q = h[N,C*D]
 *   att 3: P = x W[:F], Q = x W[F:]  ([x_i||x_j]W = P_i + Q_j, layers.py:375-376), a[C,D]
 *   e_ij   raw logit (what the reference returns as `edge_e`), i = row/dst, j = col/src
 *   alpha  = exp(sigmoid(e_ij)) / sum_row exp(sigmoid(e))      (global-max shift and the 1e-10 of
 *            utils.py:194-198 cancel / vanish: sigmoid outputs lie in (0,1))
 *   agg    = sum_j alpha_ij * mask_ij/(1-p) * V_j              (V = x W_em for AT, x W for GCN)
 *   out    = elu(agg + bias)                                   (bias: GCN only, else NULL)
 */
typedef struct {
  int32_t att;        /* 1, 2, 3 */
  int32_t C;          /* channels (--nhead) */
  int32_t D;          /* score width per channel (att 2/3); ignored for att 1 */
  int32_t Dv;         /* aggregated operand width per channel */
  int32_t training;   /* 1: apply dropout on alpha with prob `p` (layers.py:394) */
  float p;            /* dropout probability */
  uint64_t seed;      /* dropout stream; bwd must be called with the seed of its fwd */
  int32_t flags;      /* EDIS_FLAG_* (shared-operand entry points only) */
  int32_t reserved;
} edis_layer_desc;
/* edis_disga_sage_*: aggregate = plain softmax-weighted mean sum_j ad_ij x_j (no "+1" divisor):
 * gnn_type AT / GCN executed as aggregate-then-project, (sum_j ad_ij x_j) W == sum_j ad_ij (x_j W) */
#define EDIS_FLAG_PLAIN_MEAN 1
/* edis_disga_sage_bwd: the shared operand needs no gradient (layer-1 features): skip gX */
#define EDIS_FLAG_NO_GX 2
/* edis_disga_sage_bwd: run only the named passes (dst -> src -> gx, in this order on one stream;
 * none set = all).  Lets a caller time / overlap the three kernels separately. */
#define EDIS_FLAG_PHASE_DST 4
#define EDIS_FLAG_PHASE_SRC 8
#define EDIS_FLAG_PHASE_GX 16
#define EDIS_FLAG_PHASE_MASK 28

/* Forward.  Saved for backward: edge_e[E,C], stats[N,2C] (row sums: sum w, sum w*mask), hpre and,
 * for att 3, esign.
 * out / hpre: [N, C*Dv] contiguous (hpre = the aggregate BEFORE bias and ELU, out = elu(hpre + bias)).
 * workspace >= edis_graph_workspace_bytes(g, C*Dv + 2*C).
 *   esign  att 3 only, edis_disga_sign_bytes(g, d) bytes or NULL (inference: nothing is saved):
 *          one SIGN BIT per element of P_i + Q_j for every edge.  Leaky-relu is piecewise linear,
 *          so both backward passes need only lrelu'(z), never z: the destination pass reads 64 B
 *          per edge instead of re-gathering Q_j (2 KB per edge at C*D = 512), the source pass
 *          64 B instead of gathering P_i. */
int edis_disga_fwd(const edis_graph* g, const edis_layer_desc* d,
                   const float* P, int64_t ldp, const float* Q, int64_t ldq, const float* a,
                   const float* V, int64_t ldv, const float* bias,
                   float* out, float* hpre, float* edge_e, float* stats, uint8_t* esign,
                   void* workspace, int64_t workspace_bytes, void* stream);
/* bytes of the att-3 sign record for this graph / layer (0 for att 1 / 2; same for the SAGE entry) */
int64_t edis_disga_sign_bytes(const edis_graph* g, const edis_layer_desc* d);

/* Backward of edis_disga_fwd (replaces autograd through layers.py:349-416: the
 * `index_put_(accumulate)` gathers' backward and scatter_add backward).
 *   g_out[N,C*Dv]  grad wrt `out`;  g_edge_e[E,C] grad wrt the returned logits or NULL
 *   gP, gQ         grads wrt P and Q (att 1: [N,C]; att 2/3: [N,C*D]) with row strides ldgp, ldgq
 *                  (so they can be column blocks of one gradient buffer of the projection GEMM)
 *   ga[C,D]        grad wrt a (att 3), accumulated with atomics: caller zero-fills
 *   gV[N,C*Dv]     grad wrt V, row stride ldgv (grad wrt bias = column sum of gh; caller reduces)
 *   esign          the sign record the forward wrote (att 3: required; else NULL)
 *   edge_rec       scratch of edis_disga_rec_bytes(g, d) bytes handed from the dst pass to the
 *                  src pass: per edge (alpha_drop, d logit)[2C];
 *                  gh[N,C*Dv] scratch node tensor (grad wrt pre-activation)
 * workspace >= edis_graph_workspace_bytes(g, 2*C*max(D,Dv) + 2*C). */
int edis_disga_bwd(const edis_graph* g, const edis_layer_desc* d,
                   const float* P, int64_t ldp, const float* Q, int64_t ldq, const float* a,
                   const float* V, int64_t ldv, const float* bias,
                   const float* hpre, const float* edge_e, const float* stats, const uint8_t* esign,
                   const float* g_out, const float* g_edge_e,
                   float* gP, int64_t ldgp, float* gQ, int64_t ldgq, float* ga, float* gV, int64_t ldgv,
                   float* edge_rec, float* gh,
                   void* workspace, int64_t workspace_bytes, void* stream);
/* bytes of the `edge_rec` scratch for this graph / layer (same formula for the SAGE entry) */
int64_t edis_disga_rec_bytes(const edis_graph* g, const edis_layer_desc* d);
/* The two passes of edis_disga_bwd as separate calls with the same arguments (dst first, then
 * src on the same stream): destination pass over CSR (gP, ga, gh, edge_rec) and source pass
 * over CSC (gQ, gV).  edis_disga_bwd == both. */
int edis_disga_bwd_dst(const edis_graph* g, const edis_layer_desc* d,
                       const float* P, int64_t ldp, const float* Q, int64_t ldq, const float* a,
                       const float* V, int64_t ldv, const float* bias,
                       const float* hpre, const float* edge_e, const float* stats, const uint8_t* esign,
                       const float* g_out, const float* g_edge_e,
                       float* gP, int64_t ldgp, float* gQ, int64_t ldgq, float* ga, float* gV, int64_t ldgv,
                       float* edge_rec, float* gh,
                       void* workspace, int64_t workspace_bytes, void* stream);
int edis_disga_bwd_src(const edis_graph* g, const edis_layer_desc* d,
                       const float* P, int64_t ldp, const float* Q, int64_t ldq, const float* a,
                       const float* V, int64_t ldv, const float* bias,
                       const float* hpre, const float* edge_e, const float* stats, const uint8_t* esign,
                       const float* g_out, const float* g_edge_e,
                       float* gP, int64_t ldgp, float* gQ, int64_t ldgq, float* ga, float* gV, int64_t ldgv,
                       float* edge_rec, float* gh,
                       void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ SAGE neighbour mean
 * gnn_type=SAGE (layers.py:400-403 -> SageConv.forward, layers.py:96-110): the aggregated
 * operand is the raw layer input x[N,F], shared by all channels:
 *   neigh[i,c,:] = (sum_j ad_ij^c x_j) / (sum_j ad_ij^c + 1),  ad = dropped-out alpha,
 * divisor detached (layers.py:103).  Scores/softmax as in edis_disga_fwd (V = NULL there is
 * not allowed; this entry point does scoring + softmax + shared-operand aggregation).
 * neigh: [N, C*F].  stats[N,2C] as above.  */
int edis_disga_sage_fwd(const edis_graph* g, const edis_layer_desc* d,
                        const float* P, int64_t ldp, const float* Q, int64_t ldq, const float* a,
                        const float* X, int64_t ldx,
                        float* neigh, float* edge_e, float* stats, uint8_t* esign,
                        void* workspace, int64_t workspace_bytes, void* stream);
int edis_disga_sage_bwd(const edis_graph* g, const edis_layer_desc* d,
                        const float* P, int64_t ldp, const float* Q, int64_t ldq, const float* a,
                        const float* X, int64_t ldx,
                        const float* neigh, const float* edge_e, const float* stats, const uint8_t* esign,
                        const float* g_neigh, const float* g_edge_e,
                        float* gP, int64_t ldgp, float* gQ, int64_t ldgq, float* ga, float* gX,
                        float* edge_rec, float* gh,
                        void* workspace, int64_t workspace_bytes, void* stream);
/* edis_disga_sage_bwd: workspace >= edis_graph_workspace_bytes(g, W), W = 2*C*D + 2*C + F rounded up to a
 * multiple of 4. */

/* 1 if this shape runs on the 128-bit shared-operand path (F == D == 64, C in {2,4,8}), whose
 * source pass (EDIS_FLAG_PHASE_SRC) also produces gX: EDIS_FLAG_PHASE_GX is then a no-op. */
int edis_disga_sage_fused_gx(const edis_layer_desc* d);

/* ------------------------------------------------------------------ pair scoring (SSL)
 * Logits on arbitrary (i, j) pair lists, all channels [c_lo, c_hi) at once, no [M, .] temps.
 * Replaces layers.py:355-360 / 368-372 / 381-389 (`edge_auxs`).  pi/pj: int64 device arrays.
 * out[M, c_hi-c_lo].  Backward accumulates into gP/gQ/ga with vector atomics (caller
 * zero-fills or passes buffers that already hold other contributions). */
/*   psign     att 3, optional: edis_pair_sign_bytes(...) bytes; the forward records one sign bit per
 *             element of P_i + Q_j for every pair (as the layer kernels do per edge)
 *   col_perm  att 3, optional (with psign): int32[M], the pair ids sorted by j.  With both, the
 *             backward runs as two run-length passes over the sign record (rows in list order,
 *             columns through col_perm): ~100 B per pair instead of re-gathering Q_j and a 2 KB
 *             atomic per pair.  Without them (or att 1 / 2) it re-gathers and uses vector atomics. */
int edis_pair_score_fwd(const edis_layer_desc* d, int64_t n, int64_t m, const int64_t* pi,
                        const int64_t* pj, int32_t c_lo, int32_t c_hi,
                        const float* P, int64_t ldp, const float* Q, int64_t ldq, const float* a,
                        float* out, uint8_t* psign, void* stream);
int edis_pair_score_bwd(const edis_layer_desc* d, int64_t n, int64_t m, const int64_t* pi,
                        const int64_t* pj, int32_t c_lo, int32_t c_hi,
                        const float* P, int64_t ldp, const float* Q, int64_t ldq, const float* a,
                        const float* g_out, const uint8_t* psign, const int32_t* col_perm,
                        float* gP, float* gQ, float* ga, void* stream);
int64_t edis_pair_sign_bytes(const edis_layer_desc* d, int64_t m, int32_t c_lo, int32_t c_hi);

/* ------------------------------------------------------------------ fused SSL edge loss
 * loss = mean_k w_k (sigmoid(sum_c s[k,c]) - t_k)^2,  w = 1 on t != 0, else P/(M*M - P),
 * P = #(t != 0).  Replaces `torch.stack`+`sum`+`sigmoid` (pretrainer.py:730-734, 613-620) and
 * utils.adj_mse_loss (utils.py:287-298, incl. its `shape[0]**2` total on 1-D targets).
 * scores[M, Cs] (the output of edis_pair_score_fwd for the consumed channel range).
 * fwd writes loss[0] (8-byte workspace for the double accumulator), bwd writes
 * g_scores[M, Cs] = g_loss[0] * dloss/dscores (g_loss is a device scalar).
 * m_total: size of the WHOLE pair set when scores/target hold only this rank's slice of it
 * (destination-partitioned multi-GPU run; n_pos is then the positive count of the whole set and
 * the per-rank losses add up to the reference's loss); single GPU: m_total = m. */
int edis_ssl_wmse_fwd(int64_t m, int32_t cs, const float* scores, const float* target,
                      int64_t n_pos, int64_t m_total, float* loss, void* workspace,
                      int64_t workspace_bytes, void* stream);
int edis_ssl_wmse_bwd(int64_t m, int32_t cs, const float* scores, const float* target,
                      int64_t n_pos, int64_t m_total, const float* g_loss, float* g_scores,
                      void* stream);

/* ------------------------------------------------------------------ DifHead tail
 * loss = mean_i -log_softmax(logits[i, :])[label] with ONE constant label for all rows
 * (DifHeadTrainer: label == channel id, pretrainer.py:825-832 + models.py:540-541).
 * logits[N, K].  fwd writes loss[0] (8-byte workspace for the double accumulator), bwd writes
 * g_logits[N, K]. */
int edis_nll_const_label_fwd(int64_t n, int32_t k, const float* logits, int32_t label,
                             float* loss, void* workspace, int64_t workspace_bytes, void* stream);
int edis_nll_const_label_bwd(int64_t n, int32_t k, const float* logits, int32_t label,
                             const float* g_loss, float* g_logits, void* stream);

/* ------------------------------------------------------------------ stand-alone sparse ops
 * Drop-ins for utils.sp_softmax (utils.py:192-200) and utils.sp_matmul (utils.py:203-207) on
 * an arbitrary COO index list (int64 device arrays, any order), forward and backward.
 * sp_softmax keeps the reference's global-max shift and +1e-10.  denom[N] and vmax[1] are
 * scratch the caller provides (the library clears them).  values/out: [E]; mat/out: [N, F];
 * sp_matmul clears `out` / `g_mat` itself before accumulating. */
int edis_sp_softmax_fwd(int64_t n, int64_t e, const int64_t* row, const float* values,
                        float* out, float* denom, float* vmax, void* stream);
int edis_sp_softmax_bwd(int64_t n, int64_t e, const int64_t* row, const float* out,
                        const float* g_out, float* g_values, float* rowdot, void* stream);
int edis_sp_matmul_fwd(int64_t n, int64_t e, int64_t f, const int64_t* row, const int64_t* col,
                       const float* values, const float* mat, float* out, void* stream);
int edis_sp_matmul_bwd(int64_t n, int64_t e, int64_t f, const int64_t* row, const int64_t* col,
                       const float* values, const float* mat, const float* g_out,
                       float* g_values, float* g_mat, void* stream);

/* ------------------------------------------------------------------ SSL pair sampler (host)
 * Streaming replacement of `sample_train` (pretrainer.py:683-707, 552-574): merges the
 * Bernoulli hits (keys i*n+j, already collected by the caller from torch.rand row chunks so
 * the CPU RNG stream stays the reference's) with the forced positives, sorts, dedups and
 * labels against the positive set.  All HOST pointers.  pos_key sorted ascending.
 * out_key/out_label capacity n_hit + n_forced.  Returns M or <0. */
int64_t edis_merge_pairs_host(int64_t n_hit, const int64_t* hit_key, int64_t n_forced,
                              const int64_t* forced_key, int64_t n_pos, const int64_t* pos_key,
                              int64_t* out_key, float* out_label);

/* Bit-exact replay of `(torch.rand(n_draws) < thr).nonzero()` on torch's CPU generator without
 * materialising the uniforms (pretrainer.py:692 / 559 draw N x N of them per call).  HOST pointers.
 *   state   the 5056-byte blob of torch.get_rng_state() (CPUGeneratorImplState: mt19937 words,
 *           `left`, `next`); advanced IN PLACE by n_draws outputs -- torch.set_rng_state(state)
 *           then leaves the generator exactly where the reference's torch.rand would
 *   thr24   ceil(float32(thr) * 2^24): a float32 uniform is (y & 0xFFFFFF) * 2^-24
 *   out     ascending linear draw indices of the hits (k = i * N + j), capacity cap
 * Returns the hit count, or -(count) if cap is too small (state untouched), or an EDIS_ERR_*. */
int64_t edis_rand_hits_host(uint8_t* state, int64_t state_bytes, int64_t n_draws, uint32_t thr24,
                            int64_t* out, int64_t cap);

#ifdef __cplusplus
}
#endif
#endif /* EDIS_H_ */
