/*
 * twowl.h - C ABI of libtwowl_b200.so: the TwoWL (local 2-WL link prediction) message-passing
 * hot path of NguyenTrieu903/Link-Prediction-GNN as hand-written CUDA kernels for sm_100a.
 *
 * Reference interfaces replaced (file:line relative to the reference repository):
 *   TwoWL/utils.py:8-90            graph operators (degree, set_mul, check_in_set, get_ei2, blockei2,
 *                                  idx2mask, sample_block, reverse, double)
 *   TwoWL/model/model.py:37,73,77  torch_geometric.nn.GCNConv  (gcn_norm + linear + propagate + bias)
 *   TwoWL/model/model.py:38,54     torch_geometric.nn.GraphNorm (+ the Dropout / ReLU that follow it
 *                                  in Seq, model.py:36-41)
 *   TwoWL/model/model.py:53,71     nn.Embedding lookup by degree
 *   TwoWL/model/model.py:75        pair init  x[pos[:,0]] * x[pos[:,1]]
 *   TwoWL/model/model.py:78-83     readout    x[idx]; even*odd; Linear(c2, 1)
 *   TwoWL/utils.py:5,10            torch_scatter.scatter_add
 *
 * Conventions
 *   - Every pointer is a DEVICE pointer unless its name starts with h_. The library never allocates,
 *     frees or retains device memory: outputs and workspaces are caller-owned (the PyTorch caching
 *     allocator on the Python side). `*_workspace_bytes` gives the scratch size an op needs.
 *   - Index tensors at the API are int64, exactly as the reference passes them; `stride` arguments are
 *     element strides so that transposed views (get_ei2 returns cat(...).t(), utils.py:45) need no copy.
 *     Internally ids are narrowed to int32 (requires row counts < 2^31); wedge offsets stay int64.
 *   - Features are fp32 row-major [rows, C]; every feature base pointer must be 16-byte aligned and
 *     C % 4 == 0 for the vectorised kernels (C <= 1024). Other widths are TWOWL_EINVAL.
 *   - All work is enqueued on `stream` (a cudaStream_t passed as void*). No call synchronises the
 *     device; data-dependent sizes come back through device scalars the caller reads.
 *   - Return 0 on success, a positive cudaError_t, or a negative TWOWL_E*; twowl_last_error() gives
 *     a thread-local message. No exception crosses the ABI. There is no CPU fallback.
 */
#ifndef TWOWL_H_
#define TWOWL_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TWOWL_OK 0
#define TWOWL_EINVAL (-22)
#define TWOWL_ENOSPC (-28)

int twowl_version(void);
const char* twowl_last_error(void);

/* ------------------------------------------------------------------ integer operators ---------- */

/* degree (utils.py:8-10): out[v] = #{e : keys[e*stride] == v}, v in [0,num_node). out is int64[num_node]
 * and is zeroed by the call. Keys outside the range are ignored. */
int twowl_degree(const int64_t* keys, int64_t stride, int64_t n, int64_t num_node, int64_t* out,
                 void* stream);

/* Stable counting sort of the positions 0..n-1 by key = keys[i*stride] ^ key_xor:
 *   ptr[k]   (int64[num_keys+1], or NULL to skip) start of key k, ptr[num_keys] = number of in-range keys
 *   ids[...] (int32[n])          positions ordered by (key, position); out-of-range keys sort last.
 * This is the in-list / out-list build of get_ei2 (utils.py:41-44 `idx[edge[0]==i]` for all i at once)
 * and the CSR-by-target build the aggregation kernels consume. */
size_t twowl_csr_build_workspace_bytes(int64_t n, int64_t num_keys);
int twowl_csr_build(const int64_t* keys, int64_t stride, int64_t n, int64_t key_xor, int64_t num_keys,
                    int64_t* ptr, int32_t* ids, void* ws, size_t ws_bytes, void* stream);

/* out[k] = (int32)(vals[ids[k]*stride] ^ val_xor) - payload gather after twowl_csr_build. */
int twowl_gather_cols(const int32_t* ids, int64_t n, const int64_t* vals, int64_t stride, int64_t val_xor,
                      int32_t* out, void* stream);

/* get_ei2 (utils.py:36-45), step 1: off[i] = sum_{j<i} cin[j]*cout[j] for i in [0,n_node], from the two
 * CSR pointer arrays (in-list of observed edges by target, out-list of all pairs by source).
 * off[n_node] = T. */
size_t twowl_ei2_count_workspace_bytes(int64_t n_node);
int twowl_ei2_count(const int64_t* in_ptr, const int64_t* out_ptr, int64_t n_node, int64_t* off, void* ws,
                    size_t ws_bytes, void* stream);
/* step 2: write wedges t in [t_begin, t_end) as interleaved (a, b) int64 pairs: out_ab[(t-t_begin)*2+0] = a,
 * +1 = b. The [T,2] layout viewed transposed is byte-identical to the reference's return value. A rank of a
 * multi-GPU job fills only its own [t_begin, t_end). */
int twowl_ei2_fill(const int64_t* in_ptr, const int32_t* in_ids, const int64_t* out_ptr, const int32_t* out_ids,
                   const int64_t* off, int64_t n_node, int64_t t_begin, int64_t t_end, int64_t* out_ab,
                   void* stream);

/* The same wedges as two contiguous rows: out_rows[0..n) = a, out_rows[n..2n) = b, n = t_end - t_begin - the fresh contiguous
 * [2,T'] tensor blockei2's boolean indexing returns (utils.py:50). blockei2 of an index that get_ei2 made is this fill over the
 * in-lists with the blocked edges taken out: 16*T' bytes written instead of 32*T read + 16*T' written by the compaction. */
int twowl_ei2_fill_rows(const int64_t* in_ptr, const int32_t* in_ids, const int64_t* out_ptr, const int32_t* out_ids,
                        const int64_t* off, int64_t n_node, int64_t t_begin, int64_t t_end, int64_t* out_rows, void* stream);

/* idx2mask (utils.py:53-57): mask[0..num) = 0 then mask[idx[j]] = 1 (uint8). */
int twowl_mask_from_idx(const int64_t* idx, int64_t k, uint8_t* mask, int64_t num, void* stream);

/* The bounds rule of the reference's advanced indexing `x[idx]` (model.py:78 readout rows, model.py:75 pair endpoints): an id
 * in [-num, 0) wraps to id + num, anything else outside [0, num) is an IndexError there. out[i] (int64[k], contiguous) = the
 * wrapped id, or 0 for an invalid one so that no consumer kernel can read out of bounds; bad[0] (int32, zeroed by the call) =
 * the number of invalid ids, which the caller turns into an error (a device-side assertion on the Python side: no host sync). */
int twowl_index_guard(const int64_t* idx, int64_t stride, int64_t k, int64_t num, int64_t* out, int32_t* bad, void* stream);

/* Seeded uniform sampling of `count` DISTINCT non-edges (the negatives of utils.py:129-146 / datasets.py:176-197) without the
 * reference's dense N x N mask: one open-addressing hash set over the keys row*N + col holds the edges and the accepted samples;
 * slot i draws candidates from a counter-based generator keyed by (seed, i, round) and the smallest slot proposing a key wins
 * it, so the result depends on (seed, edges) only. undirected = 1: edges and samples are unordered pairs, returned with
 * row < col (the upper triangle random_split_edges keeps); 0: ordered pairs. Self loops are never sampled.
 * out_row / out_col int64[count]; done uint8[count] (or NULL) marks the slots that were filled; unresolved[0] = the number that
 * were not after `rounds` rounds (more non-edges asked for than exist, or a nearly complete graph). */
size_t twowl_nonedge_sample_workspace_bytes(int64_t n_edges, int64_t count);
int twowl_nonedge_sample(const int64_t* row, int64_t s_row, const int64_t* col, int64_t s_col, int64_t n_edges, int64_t num_nodes,
                         int64_t count, int32_t undirected, uint64_t seed, int32_t rounds, int64_t* out_row, int64_t* out_col,
                         uint8_t* done, int32_t* unresolved, void* ws, size_t ws_bytes, void* stream);

/* Per-source negatives for ranking evaluation (OGB's filtered tail corruption, ogbl-citation2 style): row i of out (int64[P*k],
 * row-major) holds k DISTINCT nodes w, uniform over the nodes allowed for src[i] (int64[P], contiguous): w != src[i] and neither
 * (src[i], w) nor (w, src[i]) is in the exclusion edge list (row, col) (strides as in twowl_nonedge_sample). Same hash table and
 * smallest-slot-wins rounds as twowl_nonedge_sample, with the claim keys (i, w) stored past the N^2 edge keys: the result depends
 * on (seed, inputs) only. Slots still unfilled after `rounds` rounds hold -1 and are counted in unresolved[0] (a source with fewer
 * than k allowed nodes, one outside [0, num_nodes), or too few rounds for a source that is adjacent to nearly every node).
 * P * k < 2^31, num_nodes < 2^31. */
size_t twowl_tail_negative_sample_workspace_bytes(int64_t n_edges, int64_t P, int64_t k);
int twowl_tail_negative_sample(const int64_t* row, int64_t s_row, const int64_t* col, int64_t s_col, int64_t n_edges, int64_t num_nodes,
                               const int64_t* src, int64_t P, int64_t k, uint64_t seed, int32_t rounds, int64_t* out,
                               int32_t* unresolved, void* ws, size_t ws_bytes, void* stream);

/* Order-preserving column selection of a [2,T] int64 matrix (blockei2 utils.py:48-50; the ei filter of
 * sample_block utils.py:62-63):
 *   mode 0: keep column t iff !mask[t]            mode 1: keep column t iff !mask[row0[t]]
 * count writes tile_off (int64[ntiles+1], ntiles = ceil(T/TWOWL_SELECT_TILE)); tile_off[ntiles] = T'.
 * fill writes out0/out1 (int64[T'] each). */
#define TWOWL_SELECT_TILE 2048
size_t twowl_select_workspace_bytes(int64_t T);
int twowl_select_count(const int64_t* row0, int64_t s0, int64_t T, const uint8_t* mask, int64_t mask_len, int mode,
                       int64_t* tile_off, void* ws, size_t ws_bytes, void* stream);
int twowl_select_fill(const int64_t* row0, int64_t s0, const int64_t* row1, int64_t s1, int64_t T,
                      const uint8_t* mask, int64_t mask_len, int mode, const int64_t* tile_off, int64_t* out0,
                      int64_t* out1, void* stream);

/* check_in_set (utils.py:22-33): out[t] = #{j : set[j] == target[t]} for values in [0, range). */
int twowl_check_in_set(const int64_t* target, int64_t st, int64_t n, const int64_t* set, int64_t m, int64_t range,
                       int32_t* counts_ws /* int32[range] */, int64_t* out, void* stream);

/* reverse (utils.py:71-78): edge = [row0^1; row1], edge_r = [row0; row1^1], both contiguous [2,T]. */
int twowl_reverse(const int64_t* row0, int64_t s0, const int64_t* row1, int64_t s1, int64_t T, int64_t* edge,
                  int64_t* edge_r, void* stream);

/* double (utils.py:81-90). edges: out[2,2M] with columns 2k=(r,c), 2k+1=(c,r). index: out[2B] = 2k,2k+1. */
int twowl_double_edges(const int64_t* r, int64_t sr, const int64_t* c, int64_t sc, int64_t M, int64_t* out,
                       void* stream);
int twowl_double_index(const int64_t* x, int64_t sx, int64_t B, int64_t* out, void* stream);

/* set_mul (utils.py:13-19): out[(i*q+j)*2+0] = a[i], +1 = b[j]. */
int twowl_set_mul(const int64_t* a, int64_t p, const int64_t* b, int64_t q, int64_t* out, void* stream);

/* int64 -> int32 narrowing copy with stride (pair table columns, index vectors). */
int twowl_narrow_i32(const int64_t* in, int64_t stride, int64_t n, int32_t* out, void* stream);

/* ------------------------------------------------------------------ aggregation ---------------- */

/* gcn_norm degree (PyG 2.3.1 gcn_norm as used by GCNConv, model.py:37) from a CSR-by-target (ptr, col):
 *   dinv[m] = (1 + #{k in CSR row (m ^ row_flip) : (col[k] ^ flip) != m, !skip_mask[col[k]]})^-1/2
 * i.e. self-loops removed, one self-loop added. A CSR row r with row_skip_mask[r] set counts as empty. */
int twowl_gcn_dinv(const int64_t* ptr, const int32_t* col, int64_t M, int32_t flip, int32_t row_flip,
                   const uint8_t* skip_mask, const uint8_t* row_skip_mask, float* dinv, void* stream);
/* same with entries removed by a per-ENTRY mask (entry_mask[k] != 0: entry k of the CSR does not exist) - the node graph
 * of one training step is the cached CSR of the whole graph minus the sampled edges (sample_block, utils.py:61-64). */
int twowl_gcn_dinv_entries(const int64_t* ptr, const int32_t* col, int64_t M, const uint8_t* entry_mask, float* dinv,
                           void* stream);
/* the same for the node rows [row_lo, row_hi) only (dinv keeps its [M] shape; the rest is untouched): one rank's node block of a
 * row-sharded step, which then all-gathers the blocks (twowl_b200.rowshard). Only entry_mask[ptr[row_lo] .. ptr[row_hi]) is read. */
int twowl_gcn_dinv_entries_rows(const int64_t* ptr, const int32_t* col, int64_t M, const uint8_t* entry_mask, int64_t row_lo,
                                int64_t row_hi, float* dinv, void* stream);
/* out[k] = mask[ids[k]] (uint8) - a per-edge mask carried to the entry order of a CSR built by twowl_csr_build. */
int twowl_gather_u8(const uint8_t* mask, const int32_t* ids, int64_t n, uint8_t* out, void* stream);

/* The one segmented gather-reduce all aggregations run through. For each output row m, with its entries
 * taken from CSR row r = m ^ row_flip (empty if row_skip_mask[r]):
 *   acc      = sum_{k in row r, kept} src_scale[s] * X[s] (* X2[mul_idx[col[k]]] if X2)   with s = col[k] ^ flip
 *              (pair_sum: X[s] + X[s ^ 1] in place of X[s])
 *   kept     = !(skip_self && s == m) && !(skip_mask && skip_mask[col[k]])
 *   out[m]   = (dst_scale ? dst_scale[m] : 1) * acc
 *            + (self_mode == 1 ? dst_scale[m]^2 * X[m] : 0)          (the GCN self-loop)
 *            + (bias ? bias : 0)                        (+ previous out[m] if accumulate)
 * Sums run in CSR order in registers: deterministic, no atomics. With a CSR built by the stable
 * twowl_csr_build the order equals the reference's scatter_add_ column order.
 * The pair-level directions of model.py:77 (reverse(), utils.py:71-78) are (flip=1,row_flip=0) for
 * edge2=[a^1;b] and (flip=0,row_flip=1) for edge2_r=[a;b^1] over ONE CSR-by-b of ei2: reverse() is folded
 * into the kernel and its two [2,T] outputs are never materialised. */
typedef struct twowl_seg_args {
  const int64_t* ptr;            /* [M+1] */
  const int32_t* col;            /* [nnz] */
  int64_t M;                     /* output rows */
  const float* X;                /* [rows_src, C] gathered rows */
  int32_t C;
  int32_t flip;                  /* 0 or 1: gathered row id = col ^ flip */
  int32_t row_flip;              /* 0 or 1: entries of output row m live in CSR row m ^ row_flip */
  const float* src_scale;        /* [rows_src] or NULL */
  const uint8_t* skip_mask;      /* indexed by col[k] (before flip) or NULL */
  const uint8_t* row_skip_mask;  /* indexed by CSR row or NULL */
  int32_t skip_self;
  int32_t self_mode;
  const float* dst_scale;        /* [M] or NULL */
  const float* bias;             /* [C] or NULL */
  const float* X2;               /* optional second factor [rows2, C] */
  const int32_t* mul_idx;        /* row of X2 = mul_idx[col[k]] */
  float* out;                    /* [M, C] */
  int32_t accumulate;
  /* optional long-row plan of this CSR (twowl_seg_plan); all NULL / 0 = every row handled by one lane group */
  const int32_t* plan_counts;    /* int32[2]: number of long rows, number of chunks */
  const int32_t* long_row;       /* int32[long_cap] */
  const int32_t* long_base;      /* int32[long_cap] */
  const int32_t* chunk_owner;    /* int32[chunk_cap] */
  float* partial;                /* fp32 [chunk_cap, C] scratch */
  int64_t chunk_cap;
  int64_t long_cap;
  int32_t pair_sum;              /* 1: gather X[s] + X[s ^ 1] (the two directions 2k / 2k+1 of one pair, utils.py:81-90);
                                    2: X has ONE row per pair that already holds that sum (twowl_conv_args.pair_sum_out): gather
                                    X[s >> 1] - the same terms in the same order, half the rows read */
  const uint8_t* entry_mask;     /* indexed by CSR ENTRY k (not by col[k]) or NULL: entries removed from a cached CSR */
  /* dual output (out2 != NULL; plain gather, flip = row_flip = 0): one pass over the 2-row blocks (s, s^1) gives
   *   out[m]  = sum src_scale[s]    * X[s]        (edge2_r's in-list sum of the pair layer, model.py:77)
   *   out2[m] = sum src_scale2[s^1] * X[s^1]      (edge2's: the same entries, the mates' rows)
   * so the two directions read H once, as 512-byte blocks. partial2 = second [chunk_cap, C] scratch when planned. */
  const float* src_scale2;
  float* out2;
  float* partial2;
  /* output rows [row_begin, row_end) only (row_end = 0: all M rows): one node block of a row-sharded multi-GPU job. ptr / col /
   * the plan / out are those of the WHOLE CSR; rows outside the range are neither read nor written. */
  int64_t row_begin;
  int64_t row_end;
  /* dual output with the mates' rows taken from a SECOND matrix: out2[m] = sum src_scale2[s^1] * X_mate[s^1] (NULL = X). One pass
   * over a node's out-list then gives both directions' gradient sums dS_f (from dO_f) and dS_r (from dO_r) of the pair layer. */
  const float* X_mate;
} twowl_seg_args;
int twowl_seg_reduce(const twowl_seg_args* h_args, void* stream);
size_t twowl_sizeof_seg_args(void);   /* binding guard: a foreign-language mirror of the struct must have this size */

/* Load balance for power-law degree: rows of a CSR longer than TWOWL_LONG_ROW entries are listed (order free)
 * and cut into chunks of TWOWL_ROW_CHUNK entries; twowl_seg_reduce then reduces the chunks with separate lane
 * groups and adds each row's partial sums in chunk order (deterministic). Built once per CSR.
 * Capacities depend on nnz only, so no device->host read is needed. */
#define TWOWL_LONG_ROW 64
#define TWOWL_ROW_CHUNK 64
int64_t twowl_seg_plan_long_cap(int64_t nnz);
int64_t twowl_seg_plan_chunk_cap(int64_t nnz);
int twowl_seg_plan(const int64_t* ptr, int64_t M, int64_t nnz, int32_t* counts /*[2]*/, int32_t* long_row,
                   int32_t* long_base, int32_t* chunk_owner, void* stream);

/* nn.Embedding forward / any row gather: out[r] = W[idx[r*stride]]  ([n, C]). */
int twowl_gather_rows(const float* W, int64_t rows_w, const int64_t* idx, int64_t stride, int64_t n, int32_t C,
                      float* out, void* stream);

/* pair init (model.py:75): out[p] = X[src[p]] * X[dst[p]]. */
int twowl_pair_init_fwd(const float* X, const int32_t* src, const int32_t* dst, int64_t R, int32_t C, float* out,
                        void* stream);

/* readout (model.py:78-83): pred[l] = sum_c H[idx[2l],c] * H[idx[2l+1],c] * w[c] + b.
 * bwd: dH must be zero-filled by the caller; rows idx[j] receive their gradient (duplicates in idx are
 * summed in index order via the sorted (key, position) list from twowl_csr_build-style sort: `order` is
 * int32[2L] positions sorted by idx value, `sorted_idx` the idx values in that order).
 * dw[C], db[1] are written (not accumulated). */
int twowl_readout_fwd(const float* H, const int64_t* idx, int64_t sidx, int64_t L, int32_t C, const float* w,
                      const float* b, float* pred, void* stream);
size_t twowl_readout_bwd_workspace_bytes(int64_t L, int32_t C);
int twowl_readout_bwd(const float* H, const int64_t* idx, int64_t sidx, int64_t L, int32_t C, const float* w,
                      const float* dpred, const int32_t* order, float* dH, float* dw, float* db, void* ws,
                      size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------ GraphNorm (+Dropout+ReLU) --- */

/* Column statistics of x[M,C] for GraphNorm (model.py:38,54; PyG 2.3.1, batch=None):
 *   stats[0:C] = mean_c(x),  stats[C:2C] = 1/sqrt(mean_c((x - mean_scale*mean)^2) + eps)
 * computed in one pass over x with shifted sums (shift = mean of the first rows) and a double-precision
 * combine using  E[(x-a*mu)^2] = Var(x) + (1-a)^2 mu^2. */
size_t twowl_graphnorm_stats_workspace_bytes(int64_t M, int32_t C);
int twowl_graphnorm_stats(const float* x, int64_t M, int32_t C, const float* mean_scale, float eps, float* stats,
                          void* ws, size_t ws_bytes, void* stream);

/* Dropout seeds (every `seed*` argument below): a counter-based hash of (seed, element index) decides each element, so the
 * backward regenerates the forward's mask from the same seed. A seed with bit 63 set is the ADDRESS (low 63 bits) of a device
 * uint64 holding the seed: a step captured as a CUDA graph keeps its seeds in device memory and refreshes them between replays. */
/* y = weight*(x - mean_scale*mean)*inv_std + bias ; then dropout(p, seed) if p > 0 ; then ReLU if relu.
 * out = y + (addend ? addend : 0)  - addend carries the other branch of the conv2s + conv2s_r sum of
 * model.py:77; it may alias out. */
int twowl_graphnorm_apply(const float* x, int64_t M, int32_t C, const float* stats, const float* weight,
                          const float* bias, const float* mean_scale, float p_drop, uint64_t seed, int32_t relu,
                          const float* addend, float* out, void* stream);

/* Backward of the fused GraphNorm+Dropout+ReLU. Given dout (gradient w.r.t. the fused output) and the saved
 * input x + stats:  dx[M,C] and dparams[4C] = (dweight, dbias, dmean_scale, column sums of dx) are written; the
 * last block is the gradient of the bias of the GCNConv that produced x, obtained without another pass. */
size_t twowl_graphnorm_bwd_workspace_bytes(int64_t M, int32_t C);
int twowl_graphnorm_bwd(const float* x, const float* dout, int64_t M, int32_t C, const float* stats,
                        const float* weight, const float* bias, const float* mean_scale, float p_drop,
                        uint64_t seed, int32_t relu, float* dx, float* dparams, void* ws, size_t ws_bytes,
                        void* stream);

/* Both GraphNorm branches of one pair layer in one pass (they share the output / the incoming gradient):
 *   apply2: out = act(drop(GN_f(xf))) + act(drop(GN_r(xr)))     - the conv2s[i](x) + conv2s_r[i](x) of model.py:77
 *   bwd2:   dxf, dxr and dparams_f[4C], dparams_r[4C] from one dout. */
int twowl_graphnorm_apply2(const float* xf, const float* xr, int64_t M, int32_t C, const float* stats_f,
                           const float* stats_r, const float* wf, const float* bf, const float* mf, const float* wr,
                           const float* br, const float* mr, float p_drop, uint64_t seed_f, uint64_t seed_r,
                           int32_t relu, float* out, void* stream);
size_t twowl_graphnorm_bwd2_workspace_bytes(int64_t M, int32_t C);
int twowl_graphnorm_bwd2(const float* xf, const float* xr, const float* dout, int64_t M, int32_t C,
                         const float* stats_f, const float* stats_r, const float* wf, const float* bf, const float* mf,
                         const float* wr, const float* br, const float* mr, float p_drop, uint64_t seed_f,
                         uint64_t seed_r, int32_t relu, float* dxf, float* dxr, float* dparams_f, float* dparams_r,
                         void* ws, size_t ws_bytes, void* stream);

/* LAST pair layer + readout (model.py:77-83): when the output of conv2s[i](x) + conv2s_r[i](x) only feeds x[idx], the two
 * GraphNorm(+Dropout+ReLU) branches are evaluated at the 2L rows idx selects, never for the whole pair table:
 *   fwd: pred[l] = sum_c hn[idx[2l],c] * hn[idx[2l+1],c] * w[c] + b,   hn[r] = act(drop(GN_f(xf[r]))) + act(drop(GN_r(xr[r])))
 *   bwd: from dpred[L]: dense dxf, dxr [M,C] (GraphNorm's statistics give every row a gradient), dparams_f / dparams_r [4C] as in
 *        twowl_graphnorm_bwd2, dw[C], db[1]. The incoming gradient is zero outside the selected rows, so the column reductions
 *        run over the 2L positions only and the dense pass reads xf, xr once. A row selected several times adds its positions in
 *        ascending order (deterministic).
 *   Masked links: a NEGATIVE id in idx[2l] / idx[2l+1] masks link l (pred[l] = 0, no gradient) - a row-sharded caller marks the
 *   links outside its row block that way; the id -2 additionally promises that every LATER link of the list is masked as well
 *   (own links packed at the front), and the kernels stop scanning there. */
int twowl_gn2_readout_fwd(const float* xf, const float* xr, int64_t M, int32_t C, const float* stats_f, const float* stats_r,
                          const float* wf, const float* bf, const float* mf, const float* wr, const float* br, const float* mr,
                          float p_drop, uint64_t seed_f, uint64_t seed_r, int32_t relu, const int64_t* idx, int64_t sidx, int64_t L,
                          const float* w, const float* b, float* pred, void* stream);
size_t twowl_gn2_readout_bwd_workspace_bytes(int64_t M, int64_t L, int32_t C);
int twowl_gn2_readout_bwd(const float* xf, const float* xr, int64_t M, int32_t C, const float* stats_f, const float* stats_r,
                          const float* wf, const float* bf, const float* mf, const float* wr, const float* br, const float* mr,
                          float p_drop, uint64_t seed_f, uint64_t seed_r, int32_t relu, const int64_t* idx, int64_t sidx, int64_t L,
                          const float* w, const float* dpred, float* dxf, float* dxr, float* dparams_f, float* dparams_r, float* dw,
                          float* db, void* ws, size_t ws_bytes, void* stream);

/* The same backward without its dense pass, for a consumer that makes dxf / dxr on the fly (twowl_pair_dw_gn): everything
 * row-sparse is done here - G[2L,C] = gradient w.r.t. hn at every selected position, head[M] / next[2L] = the chains of positions
 * that select the same row, the parameter gradients, and per branch consts[4][C] = (P, Q, sc, of) such that
 *   dx[r] = P*x[r] + Q + sc * mask(sc*x[r] + of) * sum_{positions j selecting r, ascending} G[j]
 * (consts = [f: P,Q,sc,of | r: P,Q,sc,of], 8*C floats). */
size_t twowl_gn2_readout_bwd_prepare_workspace_bytes(int64_t M, int64_t L, int32_t C);
int twowl_gn2_readout_bwd_prepare(const float* xf, const float* xr, int64_t M, int32_t C, const float* stats_f,
                                  const float* stats_r, const float* wf, const float* bf, const float* mf, const float* wr,
                                  const float* br, const float* mr, float p_drop, uint64_t seed_f, uint64_t seed_r,
                                  int32_t relu, const int64_t* idx, int64_t sidx, int64_t L, const float* w,
                                  const float* dpred, float* G, int32_t* head, int32_t* next, float* consts, float* dparams_f,
                                  float* dparams_r, float* dw, float* db, void* ws, size_t ws_bytes, void* stream);

/* Row-sharded pair table (the pair rows cut into contiguous blocks over several GPUs, SURVEY 8(e)): every column reduction
 * of the path stops at raw double sums that the caller adds over the ranks (torch.distributed all_reduce of a few KB), then the
 * second half runs on the global sums. One GPU never needs these: twowl_pair_conv / twowl_gn2_readout_bwd_prepare do both halves.
 *   twowl_graphnorm_stats_from_moments: GraphNorm (mean, inv_std) from moments[2C] = column (sum, sum of squares) over M rows
 *     (twowl_conv_args.moments, summed over ranks; M = global row count) - replaces the per-rank finalize of model.py:38.
 *   twowl_gn2_readout_bwd_rows: the row part of twowl_gn2_readout_bwd_prepare over this rank's positions -> G, head, next and
 *     colsums[6][C] (per branch sum g_y, sum g_y*n; dpred.weight; dpred.bias in column 0 of the sixth).
 *   twowl_gn2_readout_bwd_finish: from the rank-summed colsums and M_total -> consts[8C], dparams_f/r[4C], dw[C], db[1].
 *   twowl_graphnorm_bwd2_sums / _apply: twowl_graphnorm_bwd2 (non-last pair layers) cut the same way: colsums[4][C] = per branch
 *     (sum g_y, sum g_y*n) over the rank's rows; _apply = finals on the rank-summed sums with M_total + the dense dx pass. */
int twowl_graphnorm_stats_from_moments(const double* moments, int64_t M, int32_t C, const float* mean_scale, float eps,
                                       float* stats, void* stream);
size_t twowl_gn2_readout_bwd_rows_workspace_bytes(int64_t M, int64_t L, int32_t C);
int twowl_gn2_readout_bwd_rows(const float* xf, const float* xr, int64_t M, int32_t C, const float* stats_f, const float* stats_r,
                               const float* wf, const float* bf, const float* mf, const float* wr, const float* br,
                               const float* mr, float p_drop, uint64_t seed_f, uint64_t seed_r, int32_t relu, const int64_t* idx,
                               int64_t sidx, int64_t L, const float* w, const float* dpred, float* G, int32_t* head, int32_t* next,
                               double* colsums, void* ws, size_t ws_bytes, void* stream);
size_t twowl_graphnorm_bwd2_sums_workspace_bytes(int64_t M, int32_t C);
int twowl_graphnorm_bwd2_sums(const float* xf, const float* xr, const float* dout, int64_t M, int32_t C, const float* stats_f,
                              const float* stats_r, const float* wf, const float* bf, const float* mf, const float* wr,
                              const float* br, const float* mr, float p_drop, uint64_t seed_f, uint64_t seed_r, int32_t relu,
                              double* colsums, void* ws, size_t ws_bytes, void* stream);
size_t twowl_graphnorm_bwd2_apply_workspace_bytes(int32_t C);
int twowl_graphnorm_bwd2_apply(const float* xf, const float* xr, const float* dout, int64_t M, int32_t C, const float* stats_f,
                               const float* stats_r, const float* wf, const float* bf, const float* mf, const float* wr,
                               const float* br, const float* mr, float p_drop, uint64_t seed_f, uint64_t seed_r, int32_t relu,
                               const double* colsums, int64_t M_total, float* dxf, float* dxr, float* dparams_f, float* dparams_r,
                               void* ws, size_t ws_bytes, void* stream);
size_t twowl_gn2_readout_bwd_finish_workspace_bytes(int32_t C);
int twowl_gn2_readout_bwd_finish(const double* colsums, int64_t M_total, int32_t C, const float* stats_f, const float* stats_r,
                                 const float* wf, const float* bf, const float* mf, const float* wr, const float* br,
                                 const float* mr, float* consts, float* dparams_f, float* dparams_r, float* dw, float* db,
                                 void* ws, size_t ws_bytes, void* stream);

/* out[c] = sum_m x[m,c] (bias gradients). Deterministic two-level sum. */
size_t twowl_colsum_workspace_bytes(int64_t M, int32_t C);
int twowl_colsum(const float* x, int64_t M, int32_t C, float* out, void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------ dense linear layers --------- */

/* PyG Linear without bias (GCNConv.lin, model.py:37): Z[M,Co] = X[M,Ci] * W[Co,Ci]^T, fp32 in/out.
 * impl 0: SIMT FFMA tiles (exact fp32 accumulation).  impl 1: tcgen05.mma kind::tf32 with 3xTF32 split operands,
 * accumulator in TMEM (fp32-accurate to ~1e-6 relative; needs K % 32 == 0, K <= 128, N % 16 == 0, N <= 256 and the
 * split weight + one 128-row tile to fit shared memory, else TWOWL_EINVAL).  impl 2: 1 where supported, else 0.
 * bwd_input: dX[M,Ci] = dZ[M,Co] * W[Co,Ci].   bwd_weight: dW[Co,Ci] = dZ^T X (split over M, fixed order). */
int twowl_linear_fwd(const float* X, const float* W, int64_t M, int32_t Ci, int32_t Co, float* Z, int32_t impl,
                     void* stream);
int twowl_linear_bwd_input(const float* dZ, const float* W, int64_t M, int32_t Ci, int32_t Co, float* dX,
                           int32_t impl, void* stream);
size_t twowl_linear_bwd_weight_workspace_bytes(int64_t M, int32_t Ci, int32_t Co);
int twowl_linear_bwd_weight(const float* dZ, const float* X, int64_t M, int32_t Ci, int32_t Co, float* dW,
                            void* ws, size_t ws_bytes, void* stream);
/* same with dZ rows scaled on the fly: dW = (row_scale * dZ)^T X */
int twowl_linear_bwd_weight_scaled(const float* dZ, const float* row_scale, const float* X, int64_t M, int32_t Ci,
                                   int32_t Co, float* dW, void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------ fused tensor-core pair layer -- */

/* out[r,:] = sum_{s<nsrc} (row_scale_s[r] * A_s[r,:]) * B_s^T + sum_{g<ngather} tcoef_g[r] * T_g[tidx_g[r],:] + bias
 * with B_s[n][k] = W_s[n*Kd+k] (w_kn=0) or W_s[k*Nd+n] (w_kn=1), on tcgen05.mma kind::tf32 (3xTF32, TMEM accumulator),
 * one persistent warp-specialised CTA per SM. tidx < 0 = no term for that row. When `stats` is given the kernel
 * also reduces the column (sum, sum of squares) of `out` and writes GraphNorm's (mean[Nd], inv_std[Nd]) for
 * mean_scale/eps - the statistics pass of the GraphNorm that follows costs no extra read of `out`.
 * Forward of the structured pair-level GCNConv (model.py:77): A=H, row_scale=selfw, W=lin.weight, gather
 * (S W^T, centre, dinv), bias. Backward w.r.t. H: nsrc=2 over (dO_f, dO_r) with w_kn=1. */
typedef struct twowl_conv_args {
  int32_t nsrc, ngather, Kd, Nd;
  int64_t M;
  const float* A[2];          /* [M, Kd] */
  const float* row_scale[2];  /* [M] or NULL */
  const float* W[2];
  int32_t w_kn[2];
  const float* T[2];          /* [rows_T, Nd] */
  const int32_t* tidx[2];     /* [M] */
  const float* tcoef[2];      /* [M] */
  const float* bias;          /* [Nd] or NULL */
  float* out;                 /* [M, Nd] */
  float* stats;               /* [2*Nd] or NULL */
  const float* mean_scale;    /* [Nd], needed with stats */
  float eps;
  int32_t dual;               /* 1: TWO layers over the same A in one pass (both directions of model.py:77): nsrc = 1, Nd = 2*C,
                                 W[0] = [W_f; W_r] stacked ([2C, Kd], w_kn = 0), bias / mean_scale / stats / moments 2C wide; output
                                 columns [0,C) use row_scale[0], gather 0 and go to out[M,C]; columns [C,2C) use row_scale[1],
                                 gather 1 and go to out2[M,C]; the gathered tables are [rows, C]. A is read once. C % 32 == 0. */
  float* out2;                /* [M, Nd/2], dual launches */
  double* moments;            /* [2*Nd] or NULL (needs stats): the raw column (sum, sum of squares) of `out` over this call's
                                 M rows - what a row-sharded caller sums over ranks before twowl_graphnorm_stats_from_moments */
  int32_t pair_sum_out;       /* 1: `out` is [M/2, Nd] and holds result[2k] + result[2k+1] - rows 2k / 2k+1 are the two directions
                                 of one pair (utils.py:81-90) and the pair-init backward (model.py:75) only consumes their sum
                                 (twowl_seg_args.pair_sum = 2). M even, ngather = 2, no stats, no dual. */
} twowl_conv_args;
int twowl_pair_conv_supported(int32_t Kd, int32_t Nd, int32_t nsrc);
size_t twowl_pair_conv_workspace_bytes(int64_t M, int32_t Nd);
int twowl_pair_conv(const twowl_conv_args* h_args, void* ws, size_t ws_bytes, void* stream);
size_t twowl_sizeof_conv_args(void);  /* binding guard, as twowl_sizeof_seg_args */

/* Weight gradients of both pair-level linear layers in one pass over the rows (tcgen05 kind::tf32, 3xTF32, MN-major
 * operands): dWf[C,C] = (rsf * dOf)^T H, dWr[C,C] = (rsr * dOr)^T H. H is read once. C in {32, 64, 128}. */
int twowl_pair_dw_supported(int32_t C);
size_t twowl_pair_dw_workspace_bytes(int64_t M, int32_t C);
int twowl_pair_dw(const float* dOf, const float* dOr, const float* rsf, const float* rsr, const float* H, int64_t M,
                  int32_t C, float* dWf, float* dWr, void* ws, size_t ws_bytes, void* stream);

/* The same on C-column blocks of wider matrices (row pitches ld_dO / ld_H in elements): the [C,C] block of the gradients that
 * belongs to (column block of dO, column block of H). Layers wider than 128 are tiled with it. */
int twowl_pair_dw_ld(const float* dOf, const float* dOr, const float* rsf, const float* rsr, const float* H, int64_t M,
                     int32_t C, int64_t ld_dO, int64_t ld_H, float* dWf, float* dWr, void* ws, size_t ws_bytes, void* stream);

/* The same with the gradients made on the fly from the layer's OUTPUTS Of, Or (last pair layer, after
 * twowl_gn2_readout_bwd_prepare): the shared-memory pass that scales and splits the tiles first turns them into
 * dO = P*O + Q (+ the selected rows' term), writes dOf / dOr [M,C] for the later consumers, and the dense GraphNorm-backward
 * pass (2 reads + 2 writes of [M,C]) disappears. ws as twowl_pair_dw. */
int twowl_pair_dw_gn(const float* Of, const float* Or, const float* consts, const float* G, const int32_t* head,
                     const int32_t* next, float p_drop, uint64_t seed_f, uint64_t seed_r, int32_t relu, const float* rsf,
                     const float* rsr, const float* H, int64_t M, int32_t C, float* dOf, float* dOr, float* dWf, float* dWr,
                     void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------ metrics -------------------- */

/* ROC-AUC on the device (replaces pred.sigmoid().cpu().numpy() + sklearn.metrics.roc_auc_score, TwoWL/model/train.py:41-43,
 * :61-66): out[0] = AUC with tied scores sharing their average rank (= the trapezoidal area sklearn integrates),
 * out[1] = number of positives (label > 0.5), out[2] = number of negatives; AUC is NaN when one class is empty.
 * score, label: fp32[n]; out: double[3] on the device. Deterministic (radix sort + fixed-order double sums). */
size_t twowl_auc_workspace_bytes(int64_t n);
int twowl_auc(const float* score, const float* label, int64_t n, double* out, void* ws, size_t ws_bytes, void* stream);

/* Ranking metrics of the OGB link-prediction evaluators. h_ks is a HOST array of n_k cut-offs, 1 <= n_k <= TWOWL_RANK_MAX_K,
 * each >= 1. Both are deterministic: integer counts, and (MRR) double sums in a fixed two-level order. */
#define TWOWL_RANK_MAX_K 16

/* Hits@K against a shared negative set (OGB _eval_hits, ogbl-collab / ogbl-ddi): score, label fp32[n], a positive is
 * label > 0.5. out (double[n_k + 2], device) = (hits@K_1 .. hits@K_nk, n_pos, n_neg) with hits@K = #(positives with score
 * > the K-th largest negative score) / n_pos, strict >; 1.0 when n_neg < K; NaN for every K when there is no positive or any
 * score is NaN. -0.0 and +0.0 are the same score. */
size_t twowl_hits_at_k_workspace_bytes(int64_t n);
int twowl_hits_at_k(const float* score, const float* label, int64_t n, const int64_t* h_ks, int32_t n_k, double* out, void* ws,
                    size_t ws_bytes, void* stream);

/* MRR and hits@k against k negatives per positive (OGB _eval_mrr, ogbl-citation2): pos fp32[P], neg fp32[P*k] row-major (row i
 * = the k negatives of positive i). rank_i = 0.5 (#(neg_ij > pos_i) + #(neg_ij >= pos_i)) + 1; out (double[n_k + 2], device) =
 * (mean 1/rank_i, mean(rank_i <= k_1) .. mean(rank_i <= k_nk), P); every metric is NaN when P = 0 or any input is NaN. */
size_t twowl_rank_metrics_workspace_bytes(int64_t P);
int twowl_rank_metrics(const float* pos, const float* neg, int64_t P, int64_t k, const int64_t* h_ks, int32_t n_k, double* out,
                       void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------ structured wedge path ------- */

/* When ei2 is the full wedge join of (pos_edge, pred_edge) minus the wedges whose source edge is blocked
 * (what get_ei2 + blockei2 produce), the pair-level GCNConv factorises exactly through a per-node sum
 * (DESIGN.md "Factorised pair aggregation"); [2,T] is never materialised.
 * prepare: for every pair row b in [0,R) and both directions d (0: edge2=[a^1;b], 1: edge2_r=[a;b^1])
 *   centre[d][b] (int32)  node whose in-list feeds row b      dinv[d][b] = deg^-1/2
 *   selfw[d][b] = 0 if the row's own id-self-loop is among its wedges (unblocked edge) else dinv^2
 * cnt[i] = number of unblocked observed edges with target i (int32[N]). */
int twowl_wedge_prepare(const int32_t* src /*[R]*/, const int32_t* dst_e /*[E]*/, int64_t E, int64_t R, int64_t N,
                        const uint8_t* blocked /*[E] or NULL*/, const int64_t* in_ptr /*[N+1]*/, int32_t* cnt /*[N]*/,
                        int32_t* centre /*[2,R]*/, float* dinv /*[2,R]*/, float* selfw /*[2,R]*/,
                        int32_t* bnode /*[2,R]: node whose S row r feeds (backward gather), -1 if none*/, void* stream);
/* The same constants for the pair rows [row_lo, row_hi) only (even bounds: rows 2k / 2k+1 stay together): one rank's block of
 * a row-sharded step (twowl_b200.rowshard). cnt[N] is still the count over ALL live in-edges (every rank holds the int edge
 * lists); centre / dinv / selfw / bnode are [2, row_hi - row_lo]. */
int twowl_wedge_prepare_rows(const int32_t* src, const int32_t* dst_e, int64_t E, int64_t R, int64_t N, const uint8_t* blocked,
                             const int64_t* in_ptr, int64_t row_lo, int64_t row_hi, int32_t* cnt, int32_t* centre, float* dinv,
                             float* selfw, int32_t* bnode, void* stream);
/* The same for TWO ranges of pair rows [lo0, hi0) and [lo1, hi1) (even bounds, hi0 <= lo1), written one after the other into
 * [2, (hi0 - lo0) + (hi1 - lo1)] outputs: a rank's block of the row-sharded step is its slice of the observed pairs (rows < E)
 * followed by its slice of the prediction pairs (rows >= E), so that every rank carries the same share of both. */
int twowl_wedge_prepare_ranges(const int32_t* src, const int32_t* dst_e, int64_t E, int64_t R, int64_t N, const uint8_t* blocked,
                               const int64_t* in_ptr, int64_t lo0, int64_t hi0, int64_t lo1, int64_t hi1, int32_t* cnt,
                               int32_t* centre, float* dinv, float* selfw, int32_t* bnode, void* stream);
/* apply (forward):  out[b] = dinv[b]*S[centre[b]] + selfw[b]*Z[b] + bias   (centre < 0: no S term) */
int twowl_wedge_apply_fwd(const float* S, const float* Z, const int32_t* centre, const float* dinv,
                          const float* selfw, const float* bias, int64_t R, int32_t C, float* out, void* stream);
/* apply (backward): dZ[r] = selfw[r]*dO[r] + (live(a) ? dinv[r]*dS[dst_e[a]] : 0) with a = r^1 for direction 0,
 * a = r for direction 1, live(a) = a < E && !blocked[a] && dst_e[a] in [0,N). */
int twowl_wedge_apply_bwd(const float* dS, const float* dO, const int32_t* dst_e, const uint8_t* blocked, int64_t E,
                          int64_t N, const float* dinv, const float* selfw, int32_t direction, int64_t R, int32_t C,
                          float* dZ, void* stream);

/* ------------------------------------------------------------------ node-attribute input (model.py:47-51) ------ */

/* nn.Dropout(p): out[i] = x[i] / (1 - p) or 0, the mask a counter hash of (seed, i); applying it to a gradient with the same
 * seed is the backward. */
int twowl_dropout(const float* x, int64_t n, float p, uint64_t seed, float* out, void* stream);
/* bias + nn.LayerNorm(C, elementwise_affine=False, eps) + nn.Dropout(p) in one row pass (the tail of relu_lin, model.py:27-33):
 * y[m] = dropout((u - mean(u)) / sqrt(var(u) + eps)), u = z[m] + bias; stats[m] = (mean, inv_std) for the backward, which
 * returns dz = du (d bias = its column sum). */
int twowl_bias_layernorm_fwd(const float* z, const float* bias, int64_t M, int32_t C, float eps, float p, uint64_t seed, float* y,
                             float* stats, void* stream);
int twowl_bias_layernorm_bwd(const float* g, const float* z, const float* bias, const float* stats, int64_t M, int32_t C, float p,
                             uint64_t seed, float* dz, void* stream);

/* ------------------------------------------------------------------ loss + optimiser (train.py:37-39) ---------- */

/* F.binary_cross_entropy_with_logits(logits, labels) (mean reduction) forward AND backward in one pass:
 * loss[0] = mean(max(x,0) - x*y + log1p(exp(-|x|))); dlogits[i] = (sigmoid(x_i) - y_i) / n (or NULL); prob[i] = sigmoid(x_i)
 * (or NULL; what the train AUC ranks, train.py:41-43). Block partials in double, added in block order: deterministic. */
size_t twowl_bce_logits_workspace_bytes(int64_t n);
int twowl_bce_logits(const float* logits, const float* labels, int64_t n, float* loss, float* dlogits, float* prob, void* ws,
                     size_t ws_bytes, void* stream);
/* torch.optim.Adam.step() (amsgrad = False) over ONE flat fp32 buffer of n parameters; step[0] (int64, device memory: the call
 * is capturable in a CUDA graph) is the number of steps taken so far and is incremented. grad_scale (or NULL) = a device scalar
 * the gradient is multiplied by first (the 1/world of an averaged data-parallel gradient). */
int twowl_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1, float beta2,
                    float eps, float weight_decay, const float* grad_scale, int64_t* step, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TWOWL_H_ */
