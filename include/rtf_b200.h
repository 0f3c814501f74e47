/*
 * rtf_b200.h — C-ABI of librtf_b200.so: the B200 (sm_100a) kernels behind the
 * recommend-tf2.0 embedding + feature-interaction layers.
 *
 * The reference (littlemesie/recommend-tf2.0) has no native interface: its
 * boundary is the Keras Layer protocol (SURVEY.md §8b).  Each entry point below
 * names the reference call site whose stock-TensorFlow op sequence it replaces
 * (paths relative to the reference root).  The reference-side binding (ctypes
 * from the Python layer classes; a tf.load_op_library REGISTER_OP shim over the
 * same symbols) is shown in INTEGRATION.md.
 *
 * Conventions
 *  - every pointer named d_* / tables / grad / out is a DEVICE pointer unless
 *    the comment says HOST; small descriptor arrays (tables[], rows[], dims[])
 *    are HOST arrays that are copied into kernel parameters;
 *  - the caller owns every buffer, including workspaces (size query functions);
 *    the library never allocates or frees device memory and keeps no global
 *    mutable state; all work is enqueued on `stream` (a cudaStream_t) and no
 *    entry point synchronises the device;
 *  - return value: 0 = ok, negative = argument error (RTF_E_*), positive =
 *    cudaError_t from the launch;
 *  - out-of-range ids are never dereferenced: the row reads as zeros and bit 0
 *    of *d_err is set (TF CPU raises InvalidArgument; the Python layer raises
 *    when it reads the flag).
 */
#ifndef RTF_B200_H
#define RTF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTF_MAX_FIELDS 64 /* lookup slots per launch (the library chunks above it) */

#define RTF_E_ARG (-1)       /* null pointer / non-positive size */
#define RTF_E_ALIGN (-2)     /* pointer or stride not aligned for the vector path */
#define RTF_E_RANGE (-3)     /* size out of supported range */
#define RTF_E_WORKSPACE (-4) /* workspace too small */

enum { RTF_POOL_NONE = 0, RTF_POOL_SUM = 1, RTF_POOL_MEAN = 2,
       /* OR-ed into rtf_embed_fwd's pool argument (RTF_POOL_NONE only): an out-of-range id leaves its
        * output row untouched and raises no error flag (owner-gather exchange: foreign lookups) */
       RTF_POOL_SKIP_INVALID = 0x100 };
enum { RTF_OPT_NONE = 0, RTF_OPT_SGD = 1, RTF_OPT_ADAGRAD = 2, RTF_OPT_ADAM = 3 };

/* Sparse row-wise optimizer applied in place to the rows touched by a batch.
 * Keras semantics (SURVEY App. A12): Adam  m<-b1 m+(1-b1)g, v<-b2 v+(1-b2)g^2,
 * w <- w - lr_t * m/(sqrt(v)+eps), lr_t = lr*sqrt(1-b2^t)/(1-b1^t) (host passes
 * lr_t in `lr`); Adagrad acc<-acc+g^2, w<-w-lr*g/(sqrt(acc)+eps); SGD w<-w-lr*g.
 * l2 > 0 adds the regulariser gradient 2*l2*w of the touched row to g first. */
typedef struct rtf_opt {
  int32_t kind; /* RTF_OPT_* */
  float lr;
  float beta1;
  float beta2;
  float eps;
  float l2;
  /* optional DEVICE scalar: when non-NULL the kernels read the step size from *lr_dev instead of
   * `lr` — the Adam step size changes every step (bias corrections), so a training step captured
   * in a CUDA graph must not have it baked into the launch parameters */
  const float* lr_dev;
} rtf_opt;

/* library / build identification: returns the sm arch the kernels were built for (100) */
int rtf_version(int* sm_arch);

/* ---- K1: fused multi-table gather (+ sum/mean pooling over L) -----------------
 * replaces: tf.concat([embed_i(sparse[:, i]) ...], -1)   src/ctr/dlrm/model.py:45-46
 *           (+ deep_fm/model.py:53-54, autoint/model.py:46-47, din/model.py:62-74,
 *            match/sasrec/model.py:75-79) and reduce_sum(axis=1) src/match/fm/model.py:73,77
 * out[b, l, off_f + d] = W_f[ids[b,f,l], d]           (pool NONE; out is (B, L, sumD))
 * out[b, off_f + d]    = sum_l / mean_l W_f[ids[b,f,l], d]   (ascending l, fp32)
 * tables/rows/dims: HOST arrays of n_fields entries (a table may repeat).
 * ids: int32 or int64 device array addressed ids[b*sb + f*sf + l*sl].
 * out_sb: elements between consecutive samples of out (>= L*sumD or sumD). */
int rtf_embed_fwd(const float* const* tables, const int64_t* rows, const int32_t* dims,
                  int n_fields, const void* d_ids, int ids_i64, int64_t B, int L,
                  int64_t ids_sb, int64_t ids_sf, int64_t ids_sl, int pool, float* d_out,
                  int64_t out_sb, int32_t* d_err, void* stream);

/* ---- K2: deterministic embedding backward + in-place sparse optimizer ---------
 * replaces: IndexedSlices -> UnsortedSegmentSum -> ResourceApplyAdam implied by
 *           model.compile(optimizer=Adam) src/ctr/fm/train.py:49-50 (SURVEY a13)
 * sort (table,id) keys (stable LSD radix, payload = lookup position), find the
 * segments, sum each segment's gradient rows in ascending lookup position
 * (chunks of RTF_SEG_CHUNK rows; the chunk partials of every RTF_SEG_GROUP consecutive chunks
 * are added in chunk order, the group sums in group order), then apply
 * `opt` to the touched rows.  Lookup position p = (b*L + l)*n_fields + f.
 * field_table[f] (HOST) maps a field to one of n_tables distinct tables;
 * weights/state1/state2/rows/dims are HOST arrays of n_tables entries
 * (state1 = Adam m or Adagrad acc, state2 = Adam v; unused may be NULL).
 * d_grad has the layout of K1's out.  Optional outputs for inspection/tests:
 * d_uniq_key[n] (table*2^row_bits + row, ascending), d_uniq_grad[n, dim_max]
 * (the summed rows), d_num_uniq[1], and *row_bits_out (HOST). */
#define RTF_SEG_CHUNK 64
#define RTF_SEG_GROUP 64
int rtf_embed_bwd_workspace(int64_t n_lookups, int dim_max, size_t* bytes);
int rtf_embed_bwd(float* const* weights, float* const* state1, float* const* state2,
                  const int64_t* rows, const int32_t* dims, int n_tables,
                  const int32_t* field_table, int n_fields, const void* d_ids, int ids_i64,
                  int64_t B, int L, int64_t ids_sb, int64_t ids_sf, int64_t ids_sl, int pool,
                  const float* d_grad, int64_t grad_sb, const rtf_opt* opt,
                  uint32_t* d_uniq_key, float* d_uniq_grad, int32_t* d_num_uniq,
                  int* row_bits_out, void* d_workspace, size_t workspace_bytes, void* stream);

/* K2 in two halves, so that the id-only work (keys, sort, segments) can run on a side stream
 * while the forward/backward of the dense part is still computing, and only the gradient-
 * dependent half sits on the critical path.  _prepare fills the workspace; _apply consumes it
 * ONCE (same rows/dims/field_table/B/L, same workspace).  rtf_embed_bwd == prepare + apply.   */
int rtf_embed_bwd_prepare(const int64_t* rows, const int32_t* dims, int n_tables,
                          const int32_t* field_table, int n_fields, const void* d_ids,
                          int ids_i64, int64_t B, int L, int64_t ids_sb, int64_t ids_sf,
                          int64_t ids_sl, int32_t* d_num_uniq, int* row_bits_out,
                          void* d_workspace, size_t workspace_bytes, void* stream);
int rtf_embed_bwd_apply(float* const* weights, float* const* state1, float* const* state2,
                        const int64_t* rows, const int32_t* dims, int n_tables,
                        const int32_t* field_table, int n_fields, int64_t B, int L, int pool,
                        const float* d_grad, int64_t grad_sb, const rtf_opt* opt,
                        uint32_t* d_uniq_key, float* d_uniq_grad, void* d_workspace,
                        size_t workspace_bytes, void* stream);

/* ---- K4: DLRM pairwise dot interaction ------------------------------------------
 * replaces: the missing interaction at src/ctr/dlrm/model.py:48 (the file concatenates;
 *           the op is defined from the paper it cites at :7, SURVEY §8 a5)
 * X (B,F1,D) -> out[b] = [ X[b,0,:] | <X[b,i],X[b,j]> for i in 1..F1-1, j in 0..i-1 ]
 * out_cols >= D + F1(F1-1)/2 columns are written (extra columns are zero padding, so the
 * caller may round the top-MLP input width up); out_sb >= out_cols.  D % 4 == 0, F1 <= 64.
 * _bwd: d_gx[b,i,:] = sum_j S[i][j] X[b,j,:] (+ gout[b,:D] on row 0), S = sym(dZ).     */
int rtf_dot_interact_fwd(const float* d_x, int64_t B, int F1, int D, float* d_out,
                         int64_t out_sb, int out_cols, void* stream);
int rtf_dot_interact_bwd(const float* d_x, const float* d_gout, int64_t gout_sb, int64_t B,
                         int F1, int D, float* d_gx, void* stream);

/* Same interaction with the F1 rows of a sample addressed one by one: row i of sample b is
 * row_base[i] + b*row_stride[i] (HOST arrays of F1 device pointers / element strides).  Used
 * by the multi-GPU path to interact straight out of the all-to-all receive buffer (blocks
 * ordered by source rank) and to write dX rows into the send buffer of the backward
 * exchange, with no permute copy (SURVEY §8e).
 * d_xsave (optional, (B, (F1-1)*D) with sample stride xsave_sb): rows 1..F1-1 as staged, so the
 * backward can re-read them locally when the forward pulled them from peers over NVLink.   */
int rtf_dot_rows_fwd(const float* const* row_base, const int64_t* row_stride, int F1, int D,
                     int64_t B, float* d_out, int64_t out_sb, int out_cols, float* d_xsave,
                     int64_t xsave_sb, void* stream);
int rtf_dot_rows_bwd(const float* const* row_base, const int64_t* row_stride, int F1, int D,
                     int64_t B, const float* d_gout, int64_t gout_sb, float* const* grad_base,
                     const int64_t* grad_stride, void* stream);

/* ---- K1+K4 fused: gather the F embedding rows of a sample straight into shared memory
 * (one TMA bulk copy per row), append the bottom-MLP row, interact, write (B, out_cols).
 * replaces: src/ctr/dlrm/model.py:45-48 (lookup + concat + interaction) in one launch.
 * X[b,0] = d_dense[b], X[b,1+f] = tables[f][ids[b*sb + f*sf]].  All tables have dim D.
 * _bwd re-gathers X (tables must not have been updated since _fwd) and writes
 * d_gdense (B,D) and d_gemb (B, F*D) — the latter is K2's d_grad.                        */
int rtf_embed_dot_fwd(const float* const* tables, const int64_t* rows, int n_fields, int D,
                      const void* d_ids, int ids_i64, int64_t B, int64_t ids_sb, int64_t ids_sf,
                      const float* d_dense, int64_t dense_sb, float* d_out, int64_t out_sb,
                      int out_cols, int32_t* d_err, void* stream);
int rtf_embed_dot_bwd(const float* const* tables, const int64_t* rows, int n_fields, int D,
                      const void* d_ids, int ids_i64, int64_t B, int64_t ids_sb, int64_t ids_sf,
                      const float* d_dense, int64_t dense_sb, const float* d_gout,
                      int64_t gout_sb, float* d_gdense, int64_t gdense_sb, float* d_gemb,
                      int64_t gemb_sb, void* stream);

/* ---- K1+K4 over tables sharded across G GPUs (table-wise AND row-wise), NVLink peer memory ----
 * The exchange of SURVEY §8e fused into the interaction kernel: every rank keeps its table
 * shards in peer-mapped memory; the forward's TMA bulk copies pull each row from whichever GPU
 * holds it, the backward stores each dX row into the owning GPU's gradient buffer (K2's d_grad
 * there).  d_peer_tab / d_peer_gptr / d_peer_gstr are DEVICE arrays [n_fields][G] (int64):
 * shard base pointers, gradient-column base pointers and per-sample strides.  Bit f of rw_mask:
 * field f is row-wise sharded (row r on rank r % G, local row r / G); otherwise the field lives
 * on one rank and entry [f][0] is used.  rows[] (HOST) = global row counts.
 * d_peer_str != NULL ("owner gather"): the holders ran K1 for the global batch into per-rank
 * (B_global, T_g*D) buffers; d_peer_tab[f][g] = base of field f's column in rank g's buffer,
 * d_peer_str[f][g] = its sample stride, and local sample b is read at index sample0 + b.     */
int rtf_embed_dot_peer_fwd(const int64_t* d_peer_tab, const int64_t* d_peer_str, int64_t sample0,
                           int G, uint64_t rw_mask, const int64_t* rows,
                           int n_fields, int D, const void* d_ids, int ids_i64, int64_t B,
                           int64_t ids_sb, int64_t ids_sf, const float* d_dense, int64_t dense_sb,
                           float* d_out, int64_t out_sb, int out_cols, float* d_xsave,
                           int64_t xsave_sb, int32_t* d_err, void* stream);
int rtf_embed_dot_peer_bwd(const float* d_xsave, int64_t xsave_sb, const int64_t* rows,
                           int n_fields, int D, const void* d_ids, int ids_i64, int64_t B,
                           int64_t ids_sb, int64_t ids_sf, const float* d_dense, int64_t dense_sb,
                           const float* d_gout, int64_t gout_sb, float* d_gdense,
                           int64_t gdense_sb, const int64_t* d_peer_gptr,
                           const int64_t* d_peer_gstr, int G, uint64_t rw_mask, int64_t sample0,
                           void* stream);

/* ---- deterministic column sum: out[c] = sum_b rowscale[b] * x[b,c] (rowscale may be NULL) ---
 * the batch-wide reductions of weight gradients (FM w, dense FM rows, attention projections);
 * replaces the atomics-based reductions TF uses for MatMul/BiasAdd gradients.              */
int rtf_colsum_workspace(int64_t B, int cols, size_t* bytes);
int rtf_colsum(const float* d_x, int64_t x_sb, const float* d_rowscale, int64_t B, int cols,
               float* d_out, void* d_ws, void* stream);

/* ---- K3a: FM layer -------------------------------------------------------------------
 * replaces: ctr.layers.modules.FM.call  src/ctr/layers/modules.py:57-72
 * first (B,P1), w (P1), second (B,F,D) [the 2-D tensor DeepFM passes is F=M, D=1].
 *   first_batch_scalar=1, sum_d=0 : reference semantics — first order summed over the WHOLE
 *       batch (:65), out (B*D) = first + 0.5*((sum_f x)^2 - sum_f x^2)[b,d]
 *   first_batch_scalar=0          : per-sample first order (paper);  sum_d=1 also sums the
 *       second order over d -> out (B).
 * _bwd writes d_gfirst (B,P1) / d_gw (P1) / d_gsecond (B,F,D); any may be NULL.           */
int rtf_fm_layer_workspace(int64_t B, int P1, size_t* bytes);
int rtf_fm_layer_fwd(const float* d_first, int64_t first_sb, const float* d_w, int P1,
                     const float* d_second, int64_t second_sb, int F, int D, int64_t B,
                     int first_batch_scalar, int sum_d, float* d_out, void* d_ws, void* stream);
int rtf_fm_layer_bwd(const float* d_first, int64_t first_sb, const float* d_w, int P1,
                     const float* d_second, int64_t second_sb, int F, int D, int64_t B,
                     int first_batch_scalar, int sum_d, const float* d_gout, float* d_gfirst,
                     int64_t gfirst_sb, float* d_gw, float* d_gsecond, int64_t gsecond_sb,
                     void* d_ws, void* stream);

/* ---- K3b: FM model in gather form ------------------------------------------------------
 * replaces: ctr.fm.model.FM.call  src/ctr/fm/model.py:34-53 (dense one-hot (B,M) @ w, @ V^T)
 * Every feature owns one row of kp floats: columns [0,k) = its column of V, column k = its
 * w, the rest zero padding.  tables[f] (N_f,kp) for the sparse fields, d_dense_table
 * (n_dense,kp) for the dense features (scaled by their value x).
 *   A_c = sum_i x_i R_i[c];  out = sigmoid(w0 + A_k + 0.5 * sum_{c<k} (A_c^2 - sum_i x_i^2 R_i[c]^2))
 * _fwd saves A (B,kp).  _bwd writes per-sample gradient rows: d_gsparse (B, n_fields*kp) —
 * K2's d_grad — and d_gdense_rows (B, n_dense*kp) (column-sum it), and d_dz (B) (sum = dw0). */
int rtf_fm_gather_fwd(const float* const* tables, const int64_t* rows, int n_fields, int k,
                      int kp, const float* d_dense_table, int n_dense, const float* d_dense,
                      int64_t dense_sb, const void* d_ids, int ids_i64, int64_t B, int64_t ids_sb,
                      int64_t ids_sf, const float* d_w0, float* d_out, float* d_A, int32_t* d_err,
                      void* stream);
int rtf_fm_gather_bwd(const float* const* tables, const int64_t* rows, int n_fields, int k,
                      int kp, const float* d_dense_table, int n_dense, const float* d_dense,
                      int64_t dense_sb, const void* d_ids, int ids_i64, int64_t B, int64_t ids_sb,
                      int64_t ids_sf, const float* d_out, const float* d_A, const float* d_gout,
                      float* d_gsparse, float* d_gdense_rows, float* d_dz, void* stream);

/* ---- K7 / core of K6: fused short-sequence attention ------------------------------------
 * replaces: match scaled_dot_product_attention src/match/layers/modules.py:76-96 (+ the
 *           split_heads / merge transposes :63-74,122-130) and ctr
 *           _scaled_dot_product_attention src/ctr/layers/modules.py:222-240
 * q (B,Lq,H*hs), k/v (B,Lk,H*hs) addressed with element strides (sample, position); head h
 * is columns [h*hs,(h+1)*hs).  logits = q.k * scale; masked logits are REPLACED by -2^32+1
 * (a fully masked row is uniform): d_row_mask (B,Lq) blanks whole query rows (the match-side
 * (B,L,1) mask quirk, :90-91), d_key_mask (B,Lk) / causal are the conventional variants; any
 * may be NULL/0.  out (B,Lq,H*hs).  d_stat_m / d_stat_il (B,H,Lq) receive the row max and
 * 1/row-sum for the backward (both NULL for inference).  hs % 4 == 0, hs <= 128, L <= 256.
 * _bwd recomputes P; d_delta (B,H,Lq) is scratch.                                        */
int rtf_attn_fwd(const float* d_q, int64_t q_sb, int64_t q_sl, const float* d_k, int64_t k_sb,
                 int64_t k_sl, const float* d_v, int64_t v_sb, int64_t v_sl,
                 const float* d_row_mask, int64_t rm_sb, const float* d_key_mask, int64_t km_sb,
                 int causal, int B, int H, int Lq, int Lk, int hs, float scale, float* d_out,
                 int64_t o_sb, int64_t o_sl, float* d_stat_m, float* d_stat_il, void* stream);
int rtf_attn_bwd(const float* d_q, int64_t q_sb, int64_t q_sl, const float* d_k, int64_t k_sb,
                 int64_t k_sl, const float* d_v, int64_t v_sb, int64_t v_sl,
                 const float* d_row_mask, int64_t rm_sb, const float* d_key_mask, int64_t km_sb,
                 int causal, int B, int H, int Lq, int Lk, int hs, float scale,
                 const float* d_out, int64_t o_sb, int64_t o_sl, const float* d_stat_m,
                 const float* d_stat_il, const float* d_dout, int64_t do_sb, int64_t do_sl,
                 float* d_delta, float* d_dq, int64_t dq_sb, int64_t dq_sl, float* d_dk,
                 int64_t dk_sb, int64_t dk_sl, float* d_dv, int64_t dv_sb, int64_t dv_sl,
                 void* stream);

/* ---- K5: DIN local activation unit ----------------------------------------------------
 * replaces: ctr.layers.modules.AttentionLayer.call  src/ctr/layers/modules.py:149-175
 * q (B,d), k/v (B,L,d) (k may alias v), mask (B,L) float (0 = padded; NULL => every score is
 * padded, as the source does when mask is not a tensor, :164-165), W (4d) + bias (1) = the
 * Dense(1, activation) over concat([q,k,q-k,q*k]); act: 0 none, 1 relu, 2 sigmoid, 3 tanh.
 * out (B,d) = softmax(mask(act(info.W+b))) @ v, no 1/sqrt(d).  d % 4 == 0.
 * _bwd: d_gq (B,d), d_gk/d_gv (B,L,d), d_gw_rows (B,4d+1) per-sample dL/d[W|bias]
 * (column-sum it with rtf_colsum).                                                        */
int rtf_din_attn_fwd(const float* d_q, int64_t q_sb, const float* d_k, int64_t k_sb,
                     const float* d_v, int64_t v_sb, const float* d_mask, int64_t m_sb,
                     const float* d_W, const float* d_bias, int act, int64_t B, int L, int d,
                     float* d_out, int64_t o_sb, void* stream);
int rtf_din_attn_bwd(const float* d_q, int64_t q_sb, const float* d_k, int64_t k_sb,
                     const float* d_v, int64_t v_sb, const float* d_mask, int64_t m_sb,
                     const float* d_W, const float* d_bias, int act, int64_t B, int L, int d,
                     const float* d_gout, int64_t go_sb, float* d_gq, int64_t gq_sb, float* d_gk,
                     int64_t gk_sb, float* d_gv, int64_t gv_sb, float* d_gw_rows, void* stream);

/* ---- K8: sampled softmax ----------------------------------------------------------------
 * replaces: tf.nn.sampled_softmax_loss in SampledSoftmaxLayer.call
 *           src/match/layers/modules.py:54-60 (semantics: SURVEY App. A13/A14)
 * sampler: S unique log-uniform ids in [0,range_max) from a counter-based RNG (device kernel,
 * no host sync); expected counts -expm1(num_tries*log1p(-P(c))).
 * loss[b] = logsumexp([x.W[label]+b-log(te) | x.W[s_j]+b-log(se_j) (-FLT_MAX on hits)]) - true.
 * _bwd: d_gx (B,D) and d_G (B,S+1) = dL/dlogits (column 0 = true class); the weight-row
 * gradients are G^T x, scattered by K2 over ids = [labels | sampled].                      */
int rtf_log_uniform_workspace(int S, size_t* bytes);
int rtf_log_uniform_sample(uint64_t seed, int S, int64_t range_max, int64_t* d_sampled,
                           int32_t* d_num_tries, void* d_ws, void* stream);
/* same, the seed read from device memory at execution time (a step replayed from a CUDA graph
 * draws fresh candidates every replay: the host bumps *d_seed between replays)             */
int rtf_log_uniform_sample_dseed(const uint64_t* d_seed, int S, int64_t range_max,
                                 int64_t* d_sampled, int32_t* d_num_tries, void* d_ws, void* stream);
int rtf_log_uniform_expected(const int64_t* d_ids, int64_t n, int64_t range_max,
                             const int32_t* d_num_tries, float* d_out, void* stream);
int rtf_sampled_softmax_workspace(int S, int D, size_t* bytes);
int rtf_sampled_softmax_fwd(const float* d_x, int64_t x_sb, const float* d_W, const float* d_bias,
                            const int64_t* d_labels, const int64_t* d_sampled,
                            const float* d_true_exp, const float* d_samp_exp, int64_t B, int64_t N,
                            int S, int D, int remove_hits, float* d_loss, float* d_lse, void* d_ws,
                            int32_t* d_err, void* stream);
int rtf_sampled_softmax_bwd(const float* d_x, int64_t x_sb, const float* d_W, const float* d_bias,
                            const int64_t* d_labels, const int64_t* d_sampled,
                            const float* d_true_exp, const float* d_samp_exp, int64_t B, int64_t N,
                            int S, int D, int remove_hits, const float* d_lse,
                            const float* d_gloss, float* d_gx, int64_t gx_sb, float* d_G,
                            void* d_ws, void* stream);

/* K8, GEMM form for large S (same semantics as rtf_sampled_softmax_{fwd,bwd}): the (B, S) sampled
 * logits x . Ws^T come from the tensor-core GEMM (rtf_dense_gemm_nt) and these entry points do
 * the rest.  _gather: Ws (S, D) = W[sampled], cs[j] = bias[s_j] - log(samp_exp[j]).
 * _logits_fwd: true logit, accidental-hit removal, log-sum-exp -> loss, lse.
 * _logits_bwd: g0 (B) and G1 (B, S; row stride g1_ld) = d loss / d [true | sampled] logits;
 *   the caller then forms gx = G1 . Ws (rtf_dense_gemm_nn) and the weight-row gradients
 *   [g0 * x | G1^T . x] (rtf_dense_gemm_tn).  _true_gx: gx[b] += g0[b] * W[label[b]].          */
int rtf_ssm_gather(const float* d_W, const float* d_bias, const int64_t* d_sampled,
                   const float* d_samp_exp, int64_t N, int S, int D, float* d_Ws, float* d_cs,
                   int32_t* d_err, void* stream);
int rtf_ssm_logits_fwd(const float* d_logits, int64_t ld, const float* d_x, int64_t x_sb,
                       const float* d_W, const float* d_bias, const int64_t* d_labels,
                       const int64_t* d_sampled, const float* d_true_exp, const float* d_cs,
                       int64_t B, int64_t N, int S, int D, int remove_hits, float* d_loss,
                       float* d_lse, int32_t* d_err, void* stream);
int rtf_ssm_logits_bwd(const float* d_logits, int64_t ld, const float* d_x, int64_t x_sb,
                       const float* d_W, const float* d_bias, const int64_t* d_labels,
                       const int64_t* d_sampled, const float* d_true_exp, const float* d_cs,
                       int64_t B, int64_t N, int S, int D, int remove_hits, const float* d_lse,
                       const float* d_gloss, float* d_g0, float* d_G1, int64_t g1_ld, void* stream);
int rtf_ssm_true_gx(const float* d_W, const int64_t* d_labels, const float* d_g0, int64_t B,
                    int64_t N, int D, float* d_gx, int64_t gx_sb, void* stream);

/* ---- dense-layer backward epilogue (MLP either side of the path, SURVEY §8 f2) ------------
 * replaces: ReluGrad + BiasAddGrad after the Dense layers of ctr.layers.modules.DNN
 *           (src/ctr/layers/modules.py:129-135) — two passes over the (B,N) gradient become one.
 * d_g = d_gy * (d_y > 0)  (d_y NULL: no mask, d_g untouched) and d_colsum[c] = sum_b d_g[b,c]
 * in the deterministic 2-stage order of rtf_colsum.  Contiguous (B, cols), cols % 4 == 0.     */
int rtf_relu_bwd_colsum_workspace(int64_t B, int cols, size_t* bytes);
int rtf_relu_bwd_colsum(const float* d_gy, const float* d_y, int64_t B, int cols, float* d_g,
                        float* d_colsum, void* d_ws, void* stream);

/* ---- Keras binary_crossentropy on probabilities (the loss of every CTR script) --------------
 * replaces: model.compile(loss=binary_crossentropy, ...) — src/ctr/fm/train.py:49,
 *           src/ctr/deep_fm/train.py:50, src/ctr/din/train.py:103 (semantics SURVEY App. A11):
 *           pc = clip(p, 1e-7, 1-1e-7); loss = -mean(y log(pc+1e-7) + (1-y) log(1-pc+1e-7)).
 * d_y, d_p: (n) fp32.  d_loss: one float.  d_dp (n) or NULL: d loss / d p (0 where the clip
 * saturates).  One pass + a one-warp ordered sum of the 1024-element chunk partials
 * (reproducible) instead of ~30 framework elementwise launches forward + backward.          */
int rtf_bce_workspace(int64_t n, size_t* bytes);
int rtf_bce_fwd(const float* d_y, const float* d_p, int64_t n, float* d_loss, float* d_dp,
                void* d_ws, void* stream);

/* ---- Keras AUC() (ROC, interpolation, T evenly spaced thresholds; SURVEY App. A19) -----------
 * replaces: model.compile(..., metrics=[AUC()]) + model.evaluate — src/ctr/fm/train.py:50,58,67.
 * bucket(p) = max(ceilf(__fmul_rn(p, T-1)) - 1, 0); d_counts is [2][T] uint64: row 0 positives,
 * row 1 negatives PER BUCKET (not cumulative).  _update ADDS a batch of n predictions d_pred and
 * labels d_label (both fp32) to it; the caller zeroes d_counts and *d_err on reset.  An element
 * with p outside [0,1], p NaN or a label other than 0 / 1 is not counted and sets bit 0 of *d_err.
 * Shared-memory histogram per CTA, flushed with 64-bit integer atomics: the counts are exact and
 * independent of the launch order.  n == 0 launches nothing.  2 <= T <= 4096, else RTF_E_RANGE.
 * _result: tp / fp = integer suffix sums of the buckets, tpr = tp/P, fpr = fp/N (0 when P or N is
 * 0), AUC = sum_{i<T-1} (fpr[i]-fpr[i+1]) (tpr[i]+tpr[i+1]) / 2 in fp64 in a fixed order, written
 * as fp32 to *d_auc (device memory: no host sync, capturable in a CUDA graph).                  */
int rtf_auc_update(const float* d_pred, const float* d_label, int64_t n, int num_thresholds,
                   unsigned long long* d_counts, int* d_err, void* stream);
int rtf_auc_result(const unsigned long long* d_counts, int num_thresholds, float* d_auc,
                   void* stream);

/* ---- BatchNormalization of the DNN block (MLP either side of the path, SURVEY §8 f2) -------
 * replaces: tensorflow.keras.layers.BatchNormalization in training mode at the head of
 *           ctr.layers.modules.DNN (src/ctr/layers/modules.py:129-135; Keras defaults App. A9)
 *           and its gradient (FusedBatchNormV3 / FusedBatchNormGradV3).
 * x (B,C) rows ldx floats apart.  fwd: batch mean / biased variance per column (one pass, sums
 * shifted by row 0, chunk partials combined in double in chunk order — deterministic),
 * y = (x-mean)*gamma/sqrt(var+eps)+beta, moving = moving*momentum + batch*(1-momentum).
 * bwd: dbeta = sum dy, dgamma = invstd*sum dy(x-mean),
 *      dx = (dy - dbeta/B - (x-mean)*invstd^2*sum dy(x-mean)/B)*gamma*invstd.
 * NULL allowed: gamma, beta (scale/center off), y (statistics only), moving_*, dx, dgamma, dbeta. */
int rtf_bn_workspace(int64_t B, int C, size_t* bytes);
int rtf_bn_fwd(const float* d_x, int64_t ldx, int64_t B, int C, const float* d_gamma,
               const float* d_beta, float eps, float momentum, float* d_y, int64_t ldy,
               float* d_mean, float* d_invstd, float* d_moving_mean, float* d_moving_var,
               void* d_ws, size_t ws_bytes, void* stream);
int rtf_bn_bwd(const float* d_dy, int64_t lddy, const float* d_x, int64_t ldx, int64_t B, int C,
               const float* d_mean, const float* d_invstd, const float* d_gamma, float* d_dx,
               int64_t lddx, float* d_dgamma, float* d_dbeta, void* d_ws, size_t ws_bytes,
               void* stream);

/* ---- LayerNormalization of the TransformerEncoder block (either side of K7, SURVEY §8 a9) ----
 * replaces: tensorflow.keras.layers.LayerNormalization(epsilon) in
 *           src/match/layers/modules.py:173-185 (last axis, biased variance, App. A8) + gradient.
 * contiguous (rows, C), C <= 256: a warp per row (two-pass mean / centred variance in registers);
 * dgamma / dbeta are deterministic two-stage column sums.  NULL allowed: gamma, beta, dx,
 * dgamma, dbeta.                                                                               */
int rtf_layernorm_workspace(int64_t rows, int C, size_t* bytes);
int rtf_layernorm_fwd(const float* d_x, int64_t rows, int C, const float* d_gamma,
                      const float* d_beta, float eps, float* d_y, float* d_mean, float* d_rstd,
                      void* stream);
int rtf_layernorm_bwd(const float* d_dy, const float* d_x, const float* d_mean, const float* d_rstd,
                      const float* d_gamma, int64_t rows, int C, float* d_dx, float* d_dgamma,
                      float* d_dbeta, void* d_ws, size_t ws_bytes, void* stream);

/* ---- dense-layer GEMMs (MLP either side of the path, SURVEY §8 f2) --------------------------
 * replaces: the MatMul (+BiasAdd+Relu) of tensorflow.keras.layers.Dense inside
 *           ctr.layers.modules.DNN (src/ctr/layers/modules.py:114-135) and its two gradient
 *           MatMuls.  fp32 in / fp32 out on the tcgen05 tensor cores: operands are split on the
 *           fly into 3 bf16 terms and the 6 partial products weighing >= 2^-16 are accumulated
 *           in fp32 (error ~1e-7 relative, an fp32-grade GEMM; csrc/dense_gemm.cuh).
 * out[l] (M x N row-major, ldd) = act(A[l] * B[l] + bias[n]),  act = ReLU if relu else identity,
 * bias may be NULL; l = 0..batch-1 with element strides stride_* between batch items.
 *   _nn : A (M x K) row-major lda,  B (K x N) row-major ldb        forward   y = x W
 *   _nt : A (M x K) row-major lda,  B (N x K) row-major ldb        dgrad     dx = dy W^T
 *   _tn : A (K x M) row-major lda,  B (K x N) row-major ldb        wgrad     dW = x^T dy
 *         (batch > 1 = fixed split of the K = batch*K_chunk reduction; the caller sums the
 *          partial outputs in order, which keeps the result deterministic)
 * All leading dimensions / strides % 4 == 0, pointers 16-byte aligned, else RTF_E_ALIGN.     */
int rtf_dense_gemm_nn_workspace(int M, int N, int K, int batch, size_t* bytes);
int rtf_dense_gemm_nt_workspace(int M, int N, int K, int batch, size_t* bytes);
int rtf_dense_gemm_tn_workspace(int M, int N, int K, int batch, size_t* bytes);
int rtf_dense_gemm_nn(const float* d_a, int64_t lda, int64_t stride_a, const float* d_b, int64_t ldb,
                      int64_t stride_b, const float* d_bias, int relu, float* d_out, int64_t ldd,
                      int64_t stride_d, int M, int N, int K, int batch, void* d_ws, size_t ws_bytes,
                      void* stream);
int rtf_dense_gemm_nt(const float* d_a, int64_t lda, int64_t stride_a, const float* d_b, int64_t ldb,
                      int64_t stride_b, const float* d_bias, int relu, float* d_out, int64_t ldd,
                      int64_t stride_d, int M, int N, int K, int batch, void* d_ws, size_t ws_bytes,
                      void* stream);
int rtf_dense_gemm_tn(const float* d_a, int64_t lda, int64_t stride_a, const float* d_b, int64_t ldb,
                      int64_t stride_b, const float* d_bias, int relu, float* d_out, int64_t ldd,
                      int64_t stride_d, int M, int N, int K, int batch, void* d_ws, size_t ws_bytes,
                      void* stream);

/* The same GEMMs fed operands already split into three bf16 planes (csrc/dense_gemm_planes.cuh):
 * no transform warps in the mainloop, and the output is bit-identical to the fp32 entry points'
 * for the planes rtf_split_bf16x3 makes of their operands.  An operand is one bf16 tensor of
 * three planes: plane p of the element the fp32 entry point reads at offset o sits at
 * p * plane_* + o.  Strides, leading dimensions and plane strides % 8 == 0 (16 bytes) for the
 * planes, % 4 for the output; pointers 16-byte aligned; else RTF_E_ALIGN.
 *
 * rtf_split_bf16x3: planes[p * plane_stride + r * ld_out + c] = plane p of x[r * ld_in + c]:
 *   x0 = RN_satfinite(x), r = (x - x0) * 2^8, x1 = RN_satfinite(r), x2 = RN_satfinite((r - x1) * 2^8)
 *   (bf16; the GEMM mainloop's own split).  cols, ld_in, ld_out, plane_stride even.           */
int rtf_split_bf16x3(const float* d_x, int64_t rows, int cols, int64_t ld_in, uint16_t* d_planes,
                     int64_t ld_out, int64_t plane_stride, void* stream);
int rtf_dense_gemm_nn_planes_workspace(int M, int N, int K, int batch, size_t* bytes);
int rtf_dense_gemm_nt_planes_workspace(int M, int N, int K, int batch, size_t* bytes);
int rtf_dense_gemm_tn_planes_workspace(int M, int N, int K, int batch, size_t* bytes);
int rtf_dense_gemm_nn_planes(const uint16_t* d_a, int64_t lda, int64_t stride_a, int64_t plane_a,
                             const uint16_t* d_b, int64_t ldb, int64_t stride_b, int64_t plane_b,
                             const float* d_bias, int relu, float* d_out, int64_t ldd,
                             int64_t stride_d, int M, int N, int K, int batch, void* d_ws,
                             size_t ws_bytes, void* stream);
int rtf_dense_gemm_nt_planes(const uint16_t* d_a, int64_t lda, int64_t stride_a, int64_t plane_a,
                             const uint16_t* d_b, int64_t ldb, int64_t stride_b, int64_t plane_b,
                             const float* d_bias, int relu, float* d_out, int64_t ldd,
                             int64_t stride_d, int M, int N, int K, int batch, void* d_ws,
                             size_t ws_bytes, void* stream);
int rtf_dense_gemm_tn_planes(const uint16_t* d_a, int64_t lda, int64_t stride_a, int64_t plane_a,
                             const uint16_t* d_b, int64_t ldb, int64_t stride_b, int64_t plane_b,
                             const float* d_bias, int relu, float* d_out, int64_t ldd,
                             int64_t stride_d, int M, int N, int K, int batch, void* d_ws,
                             size_t ws_bytes, void* stream);

/* ---- K6: AutoInt interacting layer, fused ---------------------------------------------------
 * replaces: ctr.layers.modules.MultiHeadAttention.call on a self-attention input X (B, F, dm):
 *           Q,K,V = act(X W{q,k,v}) (no bias, src/ctr/layers/modules.py:255-270), per-head
 *           softmax(Q K^T * scale) V with no mask (:211-240), merge heads (:281-283) and, with
 *           d_w0 != NULL, relu(O + act(X W0)) (:316-323) — ONE launch per direction instead of
 *           4 tensordots + 2 transposes + 2 batched GEMMs + softmax.
 * x (B,F,dm), weights (dm, H*hs) row-major, out / gout (B,F,H*hs), all contiguous fp32.
 * act: 0 none, 1 relu, 2 sigmoid, 3 tanh.  scale: sqrt(hs) is the reference form (:235-237).
 * _supported: 1 if (F, dm, H, hs) is one of the compiled shapes (F <= 64, H*F <= 128 and
 *   (dm, H*hs, hs) in {(16,32,16), (32,32,16), (16,16,16), (16,8,8), (8,16,8), (64,64,32)});
 *   otherwise _fwd/_bwd return RTF_E_RANGE and the caller composes the layer from the
 *   projection GEMMs + rtf_attn_*.
 * _bwd: d_out = the forward's output (relu mask of the residual form; may be NULL without W0);
 *   writes d_gx (B,F,dm) and d_gw (4, dm, H*hs) = dWq|dWk|dWv|dW0 (dW0 zeros without W0), the
 *   latter reduced over the batch in a fixed order (bit-reproducible).  Workspace: _workspace. */
int rtf_autoint_layer_supported(int F, int dm, int H, int hs);
int rtf_autoint_layer_workspace(int64_t B, int dm, int HS, size_t* bytes);
int rtf_autoint_layer_fwd(const float* d_x, int64_t B, int F, int dm, const float* d_wq,
                          const float* d_wk, const float* d_wv, const float* d_w0, int H, int hs,
                          int act, float scale, float* d_out, void* stream);
int rtf_autoint_layer_bwd(const float* d_x, int64_t B, int F, int dm, const float* d_wq,
                          const float* d_wk, const float* d_wv, const float* d_w0, int H, int hs,
                          int act, float scale, const float* d_out, const float* d_gout,
                          float* d_gx, float* d_gw, void* d_ws, size_t ws_bytes, void* stream);

/* ---- a10: SASRec scoring + loss epilogue, fused with the pos / neg item gathers -------------
 * replaces: src/match/sasrec/model.py:77-79 (pos / neg Embedding lookups) and :88-96
 *           (last position, the two dot products, -log sigmoid / -log(1 - sigmoid), concat).
 * info (B, D) = att_outputs[:, -1] (row stride info_sb); pos ids (B) and neg ids (B, NEG; row
 * stride neg_sb) index the pos / neg tables (rows, D).  _fwd writes logits (B, 1+NEG) =
 * [pos | neg] and loss_rows (B) = NEG*(-log s(pos_b)) + sum_j -log(1 - s(neg_bj)); the model's
 * loss is sum_b loss_rows[b] / (2 B NEG) (finished by rtf_colsum: fixed order).  Out-of-range
 * ids read as zero rows and set *d_err.
 * _bwd: d_gloss (device scalar, may be NULL) and d_glogits (B, 1+NEG, may be NULL) are the
 * incoming gradients; writes d_ginfo (B, D) and d_gemb (B, 1+NEG, D) = ds_bj * info_b, the row
 * gradients K2 reduces per touched row (pos rows: [:,0,:], neg rows: [:,1:,:]).              */
int rtf_sasrec_score_fwd(const float* d_info, int64_t info_sb, const float* d_pos_tab,
                         int64_t pos_rows, const float* d_neg_tab, int64_t neg_rows,
                         const void* d_pos_ids, const void* d_neg_ids, int ids_i64, int64_t neg_sb,
                         int64_t B, int NEG, int D, float* d_logits, float* d_loss_rows,
                         int32_t* d_err, void* stream);
int rtf_sasrec_score_bwd(const float* d_info, int64_t info_sb, const float* d_pos_tab,
                         int64_t pos_rows, const float* d_neg_tab, int64_t neg_rows,
                         const void* d_pos_ids, const void* d_neg_ids, int ids_i64, int64_t neg_sb,
                         int64_t B, int NEG, int D, const float* d_logits, const float* d_gloss,
                         const float* d_glogits, float* d_ginfo, float* d_gemb, void* stream);

/* ---- f3: exact top-k inner-product retrieval -------------------------------------------------
 * replaces: faiss.IndexFlatIP(d).add(item_embs); D, I = index.search(user_embs, k)
 *           (src/match/fm/train.py:71-75, src/match/dssm/dssm_train.py:74-78).
 * users (B, D) row stride u_ld, items (N, D) row stride i_ld, fp32; for every user the k
 * (<= 16) items of largest inner product, best first: out_idx (B, k) int64 (-1 past N),
 * out_score (B, k) = the fp64-accumulated score rounded to fp32.  Ties: lower index first.
 * Scores come from the fp32-accurate tensor-core GEMM, the best 32 per row are re-scored in
 * fp64; bit 0 of *d_flag (caller zeroes it) is set if a row's result could not be PROVEN equal
 * to the fp64 ranking (more than 32 - k near-ties).  D % 4 == 0, N < 2^31 - 1.               */
int rtf_topk_ip_workspace(int64_t B, int64_t N, int D, int k, size_t* bytes);
int rtf_topk_ip(const float* d_users, int64_t u_ld, int64_t B, const float* d_items, int64_t i_ld,
                int64_t N, int D, int k, int64_t* d_out_idx, float* d_out_score, int32_t* d_flag,
                void* d_ws, size_t ws_bytes, void* stream);

/* ---- multi-GPU exchange, forward half as a copy kernel --------------------------------------
 * replaces: the all-to-all of pooled embeddings implied by sharding the tables that
 *           MirroredStrategy (src/ctr/fm/train.py:43) mirrors instead (SURVEY §8e).
 * Pulls the rows of this rank's B samples from the holders' owner-gathered (B_global, T_g*D)
 * buffers (same device tables of peer-mapped addresses as rtf_embed_dot_peer_fwd with
 * d_peer_str != NULL) into a LOCAL (B, n_fields*D) buffer, so that it can run on a side stream
 * behind the bottom MLP and the interaction (rtf_dot_rows_fwd) / its backward
 * (rtf_embed_dot_peer_bwd, d_xsave = this buffer) read local HBM only.                         */
int rtf_peer_pull_rows(const int64_t* d_peer_tab, const int64_t* d_peer_str, int64_t sample0, int G,
                       uint64_t rw_mask, const int64_t* rows, int n_fields, int D, const void* d_ids,
                       int ids_i64, int64_t B, int64_t ids_sb, int64_t ids_sf, float* d_out,
                       int64_t out_sb, int32_t* d_err, void* stream);

/* ---- dense optimizer steps (data-parallel replicas) ----------------------------------------
 * replaces: the ResourceApplyAdam that model.compile(optimizer=Adam(learning_rate=1e-3)) runs on
 *           every dense variable (src/ctr/fm/train.py:49-50; Keras form, SURVEY App. A12).
 * rtf_dense_adam: ONE launch over a flat fp32 buffer of n parameters (n % 4 == 0, 16-byte
 *   aligned) with its gradient and both moments; opt->lr carries the folded bias corrections
 *   lr*sqrt(1-b2^t)/(1-b1^t); same separately rounded operations as K2's row update.
 * rtf_rows_apply_dense: multi-GPU replicated small tables — K2's row update (l2 term, SGD /
 *   Adagrad / Adam) on the rows r of a contiguous (rows, dim) block whose d_touched[r] > 0, from
 *   the all-reduced summed gradients d_g (rows, dim).  Untouched rows and their state keep
 *   their values (sparse-optimizer semantics, identical on every replica).                      */
int rtf_dense_adam(float* d_w, const float* d_g, float* d_m, float* d_v, int64_t n,
                   const rtf_opt* opt, void* stream);
int rtf_rows_apply_dense(float* d_w, float* d_s1, float* d_s2, const float* d_g,
                         const float* d_touched, int64_t rows, int dim, const rtf_opt* opt,
                         void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RTF_B200_H */
