/* dggb.h -- C-ABI of the B200-native DGG hot path (libdggb.so).
 *
 * The reference (avishkarsaha/learning-adaptive-neighborhoods-for-gnns) exposes no
 * FFI of its own: its boundary is the Python nn.Module surface (SURVEY.md 8b).
 * These entry points are what a maintainer binds (ctypes / a torch extension) from
 * inside the reference's dgm.py / model.py to replace the dense ATen pipeline; each
 * one cites the reference lines it replaces.  INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host;
 *   - dense matrices are row-major fp32; graphs are int32 CSR (rowptr[N+1], col[nnz]),
 *     rows sorted by column (== the order of a coalesced torch COO tensor);
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it,
 *     nothing synchronises, nothing allocates (callers pass outputs/workspaces);
 *   - return value: DGGB_OK (0) or a negative dggb_status; no C++ exceptions cross
 *     the boundary; dggb_error_string() names a status;
 *   - buffers documented "accumulated into" must be zeroed by the caller.
 */
#ifndef DGGB_H_
#define DGGB_H_

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum dggb_status {
  DGGB_OK = 0,
  DGGB_ERR_BAD_ARG = -1,       /* null pointer / negative size */
  DGGB_ERR_BAD_SHAPE = -2,     /* unsupported dimension (e.g. H % 4 != 0 where required) */
  DGGB_ERR_UNSUPPORTED = -3,   /* unknown mode enum */
  DGGB_ERR_K_OVERFLOW = -4,    /* a row needed more than Kcap selected entries */
  DGGB_ERR_CUDA = -5,          /* a CUDA call failed; see dggb_last_cuda_error() */
  DGGB_ERR_WORKSPACE = -6      /* workspace too small */
} dggb_status;

int dggb_version(void);                     /* ABI version, currently 2 */
const char* dggb_error_string(int status);
int dggb_last_cuda_error(void);             /* cudaError_t of the last DGGB_ERR_CUDA */
int dggb_build_arch(void);                  /* 1000 == compiled for sm_100a */
long long dggb_kernel_launches(void);       /* kernels launched by this library so far */

/* ------------------------------------------------------------------------------------
 * Graph plumbing.  Replaces (A.to_dense() + I).to_sparse().coalesce()
 * (model.py:1249-1264, 171-176, 389-392, 710-715, 1381-1392) and the COO->dense
 * scatters (dgm.py:1787-1788, 1626-1627).
 * ---------------------------------------------------------------------------------- */

/* rowptr[N+1] from the row indices of a COALESCED COO (int64, sorted). */
int dggb_coo_rows_to_rowptr(const int64_t* row, int64_t nnz, int32_t n, int32_t* rowptr, void* stream);

/* int64 -> int32 column indices. */
int dggb_cast_i64_i32(const int64_t* src, int32_t* dst, int64_t n, void* stream);

/* erow[e] = row of CSR entry e (the COO row array, int32). */
int dggb_csr_expand_rows(const int32_t* rowptr, int32_t n, int32_t* erow, void* stream);

/* CSR + I: per row, add 1.0 to an existing diagonal entry or insert a new one.
 * Two phases so the caller can size the output: phase 1 writes out_rowptr[N+1];
 * the caller reads out_rowptr[N] (nnz_out) and allocates; phase 2 fills col/val. */
int dggb_add_self_loops_count(const int32_t* rowptr, const int32_t* col, int32_t n,
                              int32_t* out_rowcount /* [N+1], exclusive-scanned in place */, void* stream);
int dggb_add_self_loops_fill(const int32_t* rowptr, const int32_t* col, const float* val, int32_t n,
                             const int32_t* out_rowptr, int32_t* out_col, float* out_val, void* stream);

/* ------------------------------------------------------------------------------------
 * class DGG edge ranker + degree estimator + soft first-k (dgm.py:1781-1810; a4, A.1)
 *
 *   y      = x_enc * We^T            (the caller's GEMM; Linear(h,h) of dgm.py:1784 is
 *                                     linear, so We(x_u - x_v) + be == y_u - y_v + be)
 *   R_e    = sigmoid( sum_c LeakyReLU_0.01( y[u,c] - y[v,c] + be[c] ) )        (1783-1786)
 *   [ablation: R_e = sigmoid(R_e + noise_e), noise_e in U(-1,1)]                (1933-1935)
 *   s_i    = sum_{e in row i} R_e ;  k_i = LeakyReLU_0.01(deg_w * s_i + deg_b)   (1791-1792)
 *   r_e    = 0-based descending rank of R_e inside its row (ties: lower column first)
 *   out_e  = R_e * ( (1 - 0.5*(1 + tanh(r_e - k_i))) + 1 )                       (1798-1810)
 *   [hard_k >= 0: out_e = r_e < hard_k ? R_e : 0 and k is not computed]          (1943-1945)
 *
 * Two launches: an edge-parallel score pass (balanced under power-law degrees) and a
 * warp-per-row rank pass.  The dense N x N scatter, the N-long row sort and the un-sort scatter of the reference
 * are not performed: off-support entries are exact zeros that sort last, so the rank
 * inside the row's own edges is the rank in the dense row.
 * Requires H % 4 == 0.  nnz == 0 is allowed (erow, col, R, rank, out, and g_out in the backward, may then be
 * NULL): every row gets s = 0 and k = LeakyReLU(deg_b), and the backward adds nothing.
 * ---------------------------------------------------------------------------------- */
int dggb_dgg_edge_fwd(const int32_t* rowptr, const int32_t* erow /* [E] row of each entry */,
                      const int32_t* col, int32_t n, int32_t nnz, int32_t h,
                      const float* y /* [N,H] */, const float* be /* [H] */,
                      const float* deg_w /* [1] */, const float* deg_b /* [1] */,
                      const float* ablation_noise /* [E] or NULL */, int32_t hard_k /* <0: soft */,
                      float* R /* [E] out (post-noise value) */, int32_t* rank /* [E] out */,
                      float* s /* [N] out */, float* k /* [N] out */, float* out /* [E] out */,
                      int32_t* long_ws /* NULL, or [N+1] scratch with long_ws[0] == 0: rows longer than 1024
                                          entries (power-law hubs) are listed there and ranked by a third,
                                          grid-wide launch instead of one warp each */,
                      void* stream);

/* Backward of the above w.r.t. y, be, deg_w, deg_b given g_out = dL/d out.
 * dy[N,H], dbe[H], ddeg[2] (= {d deg_w, d deg_b}) are ACCUMULATED INTO; ds_ws[N] is scratch.
 * The per-edge pre-activations are recomputed from y, never stored. */
int dggb_dgg_edge_bwd(const int32_t* rowptr, const int32_t* erow, const int32_t* col, int32_t n,
                      int32_t nnz, int32_t h,
                      const float* y, const float* be, const float* deg_w, const float* deg_b,
                      const float* ablation_noise, int32_t hard_k,
                      const float* R, const int32_t* rank, const float* s, const float* k,
                      const float* g_out /* [E] */, float* ds_ws /* [N] scratch */,
                      float* dy, float* dbe, float* ddeg, void* stream);

/* Single-launch variants of the two calls above for graphs whose longest row has at most 512 entries
 * (max_row_nnz: the caller's cached max over rows of rowptr[i+1]-rowptr[i]; Cora / Citeseer / Pubmed qualify).
 * A block owns the rows that start inside its slice of the entry range, keeps their scores (fwd) / ds (bwd) in
 * shared memory and runs both phases back to back.  Same arguments.  R and rank are the two-launch results bit for
 * bit; s, k, out and the gradients differ from them by the summation order of the row sums (and of the atomics).
 * Return DGGB_ERR_UNSUPPORTED when max_row_nnz > 512 or nnz == 0: call the two-launch entry point instead.
 * DGGB_FUSED_EPB (read per call; values below 1 are ignored) sets the smallest number of entries per block.
 *
 * Training goes through the _mask pair.  The forward also stores what the backward would otherwise recompute from y:
 *   branch_mask [E, ceil(H/32)] uint32: bit c % 32 of word c / 32 is set when pre_c = y_u - y_v + be > 0;
 *   r1 [E]: the pre-noise sigmoid(z), written only when ablation_noise != NULL (then it is required with the mask).
 * Both may be NULL (inference).  The backward reads them instead of y and be (8 B per entry at H = 64 instead of two
 * 4 H-byte row gathers) and gives the gradients of the unmasked pair up to the order of the atomics.
 *
 * dggb_dgg_edge_bwd_fused, without a mask to read, runs the two-launch dggb_dgg_edge_bwd (same arguments, same
 * accumulate-into contract, any dbe alignment); it stays for callers of this ABI. */
int dggb_dgg_edge_fwd_fused_mask(const int32_t* rowptr, const int32_t* erow, const int32_t* col, int32_t n,
                                 int32_t nnz, int32_t max_row_nnz, int32_t h, const float* y, const float* be,
                                 const float* deg_w, const float* deg_b, const float* ablation_noise,
                                 int32_t hard_k, float* R, int32_t* rank, float* s, float* k, float* out,
                                 uint32_t* branch_mask /* [E, ceil(H/32)] out, or NULL */,
                                 float* r1 /* [E] out when ablation_noise != NULL, or NULL */,
                                 float* zero_ws, int64_t zero_count, void* stream);
int dggb_dgg_edge_bwd_fused_mask(const int32_t* rowptr, const int32_t* erow, const int32_t* col, int32_t n,
                                 int32_t nnz, int32_t max_row_nnz, int32_t h, const float* deg_w,
                                 const float* deg_b, const float* ablation_noise, int32_t hard_k, const float* R,
                                 const int32_t* rank, const float* s, const float* k,
                                 const uint32_t* branch_mask /* [E, ceil(H/32)] from the forward */,
                                 const float* r1 /* [E] from the forward when ablation_noise != NULL, or NULL */,
                                 const float* g_out, float* ds_ws, float* dy, float* dbe, float* ddeg,
                                 void* stream);
int dggb_dgg_edge_fwd_fused(const int32_t* rowptr, const int32_t* erow, const int32_t* col, int32_t n,
                            int32_t nnz, int32_t max_row_nnz, int32_t h, const float* y, const float* be,
                            const float* deg_w, const float* deg_b, const float* ablation_noise,
                            int32_t hard_k, float* R, int32_t* rank, float* s, float* k, float* out,
                            float* zero_ws /* or NULL: zero_count floats cleared by this launch (the
                                              backward's dy|dbe|ddeg|ds buffer), saving a fill launch */,
                            int64_t zero_count, void* stream);
int dggb_dgg_edge_bwd_fused(const int32_t* rowptr, const int32_t* erow, const int32_t* col, int32_t n,
                            int32_t nnz, int32_t max_row_nnz, int32_t h, const float* y, const float* be,
                            const float* deg_w, const float* deg_b, const float* ablation_noise,
                            int32_t hard_k, const float* R, const int32_t* rank, const float* s,
                            const float* k, const float* g_out, float* ds_ws, float* dy, float* dbe,
                            float* ddeg, void* stream);

/* ------------------------------------------------------------------------------------
 * select_top_k of DGG_LearnableK_debug, mode "k_times_edge_prob" (dgm.py:1402-1421; a10, A.2)
 * on CSR rows with an externally estimated k [N]:
 *   out_e = score_e * (1 - 0.5*(1 + tanh(r_e - k_i))),  r_e = descending in-row rank of score_e.
 * Exact zeros (tanh saturated) stay in the support as explicit zeros.
 * mode 1 = "k_only" (dgm.py:1423-1435): out_e = fk(r_e - k_i), the scores only decide the order (no gradient).
 * bwd: dscore_e = g_e * fk_e;  dk_i = 0.5 * sum_e g_e score_e sech^2(r_e - k_i)  (both OVERWRITTEN;
 *      mode 1: dscore = 0, dk_i = 0.5 * sum_e g_e sech^2(r_e - k_i)).
 * ---------------------------------------------------------------------------------- */
int dggb_row_firstk_fwd(const int32_t* rowptr, int32_t n, const float* score /* [E] */,
                        const float* k /* [N] */, int32_t mode /* 0 k_times_edge_prob, 1 k_only */,
                        int32_t* rank /* [E] out */, float* out /* [E] out */,
                        int32_t* long_ws /* NULL or [N+1] zero-headed scratch, see dggb_dgg_edge_fwd */,
                        void* stream);
int dggb_row_firstk_bwd(const int32_t* rowptr, int32_t n, const float* score, const float* k, int32_t mode,
                        const int32_t* rank, const float* g_out, float* dscore /* [E] */,
                        float* dk /* [N] */, void* stream);

/* ------------------------------------------------------------------------------------
 * edge_prob_net of DGG_LearnableK_debug (dgm.py:1596-1727; a8), one fused kernel per direction.
 *
 * The first Linear of edge_encode acts on the concatenation [x_u ; x_v ; extra], so it splits into per-NODE
 * projections computed once by a tall GEMM (p_uv = x_enc [W1_u ; W1_v]^T, [N, ldp], u half in columns [0, w),
 * v half in [w, 2w)) plus a per-edge rank-M update:
 *     score_e = sigmoid( b2 + sum_c w2[c] * act( p_uv[u, c] + p_uv[v, w + c] + b1[c] + sum_m wx[c, m] extra_m(e) ) )
 * act = LeakyReLU(slope) (slope == 1: identity).  flags select the extra features, in this order:
 *     1 (DGGB_EX_VAL)   extra = (A_uv)                                  "u-v-A_uv"      dgm.py:1628-1644
 *     2 (DGGB_EX_DEG)   extra = (deg[u], deg[v])                         "u-v-deg"       dgm.py:1645-1670
 *     2|4 (.. | DIST)   extra = (deg[u], deg[v], exp(-dist_scale |xe_u - xe_v|))  "u-v-deg-dist"  1671-1702
 *     0                 no extras: "edge_conv" with p_uv = xe [W_phi - W_theta ; W_theta]^T, b1 = b_theta + b_phi,
 *                       slope = 1, w2 / b2 = edge_conv_encode                              dgm.py:1703-1719
 *     8 (DGGB_DIST_ONLY) score_e = exp(-dist_scale |xe_u - xe_v|_2), nothing else is read   "u-v-dist"  1618-1623
 * wx: [w, M] row-major (the last M columns of edge_encode.0.weight).  w, hx multiples of 4 and <= 512.
 * bwd: g_score = dL/dscore; d_p_uv [N, ldp], d_xe [N, hx], d_wx, d_b1, d_w2, d_b2 are ACCUMULATED INTO (zero them);
 * pre-activations are recomputed from the gathered rows, no [E, w] tensor is stored.  d_xe may be NULL (distance
 * feature treated as a constant) except with DGGB_DIST_ONLY.
 * ---------------------------------------------------------------------------------- */
#define DGGB_EX_VAL 1
#define DGGB_EX_DEG 2
#define DGGB_EX_DIST 4
#define DGGB_DIST_ONLY 8
int dggb_edge_mlp_fwd(const int32_t* erow, const int32_t* col, int32_t nnz, int32_t w, int32_t ldp,
                      const float* p_uv, const float* xe /* [N,hx] or NULL */, int32_t hx,
                      const float* edge_val /* [E] or NULL */, const float* deg /* [N] or NULL */,
                      const float* wx, const float* b1, const float* w2, const float* b2, float slope,
                      float dist_scale, int32_t flags, float* score /* [E] out */, void* stream);
int dggb_edge_mlp_bwd(const int32_t* erow, const int32_t* col, int32_t nnz, int32_t w, int32_t ldp,
                      const float* p_uv, const float* xe, int32_t hx, const float* edge_val, const float* deg,
                      const float* wx, const float* b1, const float* w2, const float* b2, float slope,
                      float dist_scale, int32_t flags, const float* score, const float* g_score,
                      float* d_p_uv, float* d_xe, float* d_wx, float* d_b1, float* d_w2, float* d_b2,
                      void* stream);

/* ------------------------------------------------------------------------------------
 * normalize_adj: Ahat_ij = A_ij * s_i^-1/2 * s_j^-1/2 with s = ROW sums on both sides
 * (model.py:1215-1218, 146-149, 687-690, 1347-1350; dgm.py:1172-1175; a13, A.6).
 * Replaces diag + two dense N^3 torch.mm with O(nnz) work.
 * ---------------------------------------------------------------------------------- */
int dggb_sym_normalize_fwd(const int32_t* rowptr, const int32_t* col, const float* val, int32_t n,
                           float* dinv /* [N] out: s^-1/2 */, float* out /* [E] */, void* stream);
/* dval_e = g_e*a_i*a_j - 0.5 * s_i^-3/2 * T_i,  T_i = sum over entries whose row OR column is i
 * of g*val*a_other.  t_ws [N] is scratch and must be zeroed by the caller. */
int dggb_sym_normalize_bwd(const int32_t* rowptr, const int32_t* col, const float* val, int32_t n,
                           const float* dinv, const float* g /* [E] */, float* t_ws /* [N] zeroed */,
                           float* dval /* [E] out */, void* stream);

/* ------------------------------------------------------------------------------------
 * CSR SpMM  Y = A X  -- replaces torch.mm(adj_dense, x) (model.py:594, 67) and the
 * dense adj @ x of PyG DenseGraphConv (model.py:128-129).  128-bit gathers when F%4==0.
 * row_scale (may be NULL): Y_i *= row_scale[i]  (SAGE mean: 1/clamp(rowsum,1)).
 * ---------------------------------------------------------------------------------- */
int dggb_spmm_csr_fwd(const int32_t* rowptr, const int32_t* col, const float* val, int32_t n,
                      const float* x /* [Ncols,F] */, int32_t f, const float* row_scale,
                      float* y /* [N,F] */, void* stream);
/* Backward: dval_e = rs_i * <dY_i, X_j> (skipped if dval NULL); dX_j += val_e * rs_i * dY_i
 * (dX ACCUMULATED INTO via vector atomics; skipped if NULL). */
int dggb_spmm_csr_bwd(const int32_t* rowptr, const int32_t* col, const float* val, int32_t n,
                      const float* x, int32_t f, const float* row_scale, const float* dy,
                      float* dval, float* dx, void* stream);

/* ------------------------------------------------------------------------------------
 * GATConv_DGG (model.py:534-577; a19, SURVEY A.5) and GATConv (model.py:489-531) aggregation, all heads in one
 * launch.  hd [N, ldh]: head k owns columns [k F, (k+1) F); pq [N, heads, 2] = (h_i . a[:F], h_i . a[F:]);
 * the CSR (rowptr, col) is the listed edge set, adj_val [E] the DGG weights A_ij on it (NULL: 1).
 *   s_e = LeakyReLU_alpha(p_i + q_j) * A_ij ;  m_i = max(0, max_e s_e) ;  x_e = exp(s_e - m_i) ;  em_i = exp(-m_i)
 *   Z_i = sum_e (x_e - em_i) + bg_count * em_i
 *   out_i = [ sum_e (keep_e x_e - em_i) hd_j + em_i htot ] / Z_i + bias
 * -- the closed form of the reference's DENSE softmax: its mask is applied by multiplication, so a non-listed pair
 * has logit -1e20 * 0 = -0.0 and every row's softmax runs over all bg_count = N columns.  bg_count == 0 is the plain
 * masked softmax of GATConv (em := 0, m_i = max_e s_e).  keep [heads, E] (NULL: 1): attention-dropout multipliers
 * on the listed entries (the background keeps its expectation).  htot [heads F] = column sums of hd.
 * F % 4 == 0, F <= 512.  m_out / z_out [N, heads] are saved for the backward.
 * bwd: d_hd [N, ldh], d_pq [N, heads, 2], d_adj_val [E] (or NULL), d_htot [heads F] (or NULL) ACCUMULATED INTO.
 * ---------------------------------------------------------------------------------- */
int dggb_gat_aggregate_fwd(const int32_t* rowptr, const int32_t* col, int32_t n, int64_t nnz, int32_t heads,
                           int32_t f, const float* hd, int32_t ldh, const float* pq, const float* adj_val,
                           const float* keep, const float* htot, const float* bias, float alpha, float bg_count,
                           float* out /* [N, ldo] */, int32_t ldo, float* m_out, float* z_out, void* stream);
int dggb_gat_aggregate_bwd(const int32_t* rowptr, const int32_t* col, int32_t n, int64_t nnz, int32_t heads,
                           int32_t f, const float* hd, int32_t ldh, const float* pq, const float* adj_val,
                           const float* keep, const float* bias, float alpha, float bg_count, const float* out,
                           const float* g_out, int32_t ldo, const float* m_in, const float* z_in, float* d_hd,
                           float* d_pq, float* d_adj_val, float* d_htot, void* stream);

/* Edge-parallel variants of the two calls above for short-row graphs (citation graphs: ~5 entries per row): groups of
 * lanes walk runs of 8 consecutive entries instead of one warp per row -- ~10x fewer instructions at Pubmed shape and
 * perfectly balanced under power-law degrees.  y MUST BE ZEROED by the caller (rows cut by a run boundary are combined
 * with vector reductions); erow = row of every entry (dggb_csr_expand_rows).  F % 4 == 0, F <= 512. */
int dggb_spmm_edge_fwd(const int32_t* rowptr, const int32_t* erow, const int32_t* col, const float* val, int32_t n,
                       int64_t nnz, const float* x, int32_t f, const float* row_scale, float* y, void* stream);
int dggb_spmm_edge_bwd(const int32_t* erow, const int32_t* col, const float* val, int64_t nnz, const float* x,
                       int32_t f, const float* row_scale, const float* dy, float* dval, float* dx, void* stream);

/* ------------------------------------------------------------------------------------
 * SpMM with the conv layer's dense part folded in -- GCNConv relu((A x) W) (model.py:594-598) and the GCNII layer
 * theta * (s W) + (1 - theta) * s, s = (1 - alpha) A h + alpha h0 (model.py:32-44, 65-77) -- one launch per
 * direction instead of SpMM + axpby + library GEMM + axpby + add + relu:
 *     s_i = c1 * rs_i * sum_e a_e x[col_e] + c2 * h0_i ;   y_i = act(theta * (s_i W) + beta * s_i + resid_i)
 * W [Fin, Fout] row-major (held in shared memory); h0 / resid / row_scale / s_out may be NULL; relu != 0: act = ReLU.
 * Fin % 4 == 0, Fin <= 128, Fout <= 128; beta != 0 requires Fout == Fin.  s_out [N, Fin] receives theta * s: what the
 * weight gradient dW = (theta s)^T dY needs (dggb_gemm_tn_splitk).
 * bwd (gy = dL/dy already masked by the ReLU): ds_i = theta * (gy_i W^T) + beta * gy_i  -> ds_out [N, Fin] =
 * ds_scale * ds (d h0 = c2 * ds: pass ds_scale = c2), dval_e = rs_i c1 <ds_i, x_col> (OVERWRITTEN; NULL: skipped),
 * dx_col += a_e rs_i c1 ds_i (ACCUMULATED).  zero_ws / zero_count: optional fp32 buffer cleared by this launch (the
 * split-K accumulator of the weight gradient that follows).  relu_y [N, Fout] (or NULL): the forward's ReLU output --
 * gy is then the UNMASKED upstream gradient and the kernel applies the threshold itself; gy_masked [N, Fout] (or NULL)
 * receives the masked gradient (what the weight gradient needs).
 * out_keep [N, Fout] (or NULL, both directions): dropout multipliers (0 or 1 / (1 - p)) applied to the layer OUTPUT,
 * y = act(...) * out_keep -- the F.dropout in front of the NEXT GCNII layer (model.py:725) and its backward are two
 * launches per layer and direction otherwise; the backward takes gy = dL/dy of that dropped output.
 * accumulate (bwd): bit 0: dval += instead of =, bit 1: ds_out += instead of = -- the layers of a deep stack that share
 * the adjacency values / h0 (GCNII: all 64) sum their gradients in place instead of through 2 x 63 add launches.
 * ---------------------------------------------------------------------------------- */
int dggb_spmm_gemm_fwd(const int32_t* rowptr, const int32_t* col, const float* val, int32_t n, const float* x,
                       int32_t fin, const float* row_scale, const float* h0, float c1, float c2, const float* w,
                       int32_t fout, float theta, float beta, const float* resid, int32_t relu,
                       const float* out_keep, float* y, float* s_out, void* stream);
int dggb_spmm_gemm_bwd(const int32_t* rowptr, const int32_t* col, const float* val, int32_t n, const float* x,
                       int32_t fin, const float* row_scale, float c1, const float* w, int32_t fout, float theta,
                       float beta, const float* gy, float* dval, float* dx, float* ds_out, float ds_scale,
                       float* zero_ws, int64_t zero_count, const float* relu_y, float* gy_masked,
                       const float* out_keep, int32_t accumulate, void* stream);

/* A STACK of GCNII layers that share the adjacency and h0 in ONE cooperative launch (small graphs: one warp per row,
 * every CTA resident, grid barrier between layers): y[k] = ReLU(theta_k (s_k W_k) + (1 - theta_k) s_k) * keep[k],
 * s_k = c1 (A y[k-1]) + c2 h0, y[-1] = x0  (GraphConvolution, model.py:65-77, as GCNII_DGG calls it 62 times behind its
 * last DGG layer, model.py:722-729).  w_host_ptrs / theta_host are HOST arrays of `layers` device pointers ([f, f] each)
 * and floats; y / s_out: [layers, n, f] (s_out receives theta_k s_k, the weight gradient's left operand, or NULL);
 * keep: [layers, n, f] or NULL; barrier_zeroed: one zeroed uint32.  f in {32, 64, 128}, layers <= 96.  Returns
 * DGGB_ERR_UNSUPPORTED when the grid cannot be resident at once (n > dggb_gcnii_stack_max_rows(f), ~4 700 rows at
 * f = 64): run the layers one launch each (dggb_spmm_gemm_fwd).  The backward is per layer (dggb_spmm_gemm_bwd with its accumulate flags). */
int32_t dggb_gcnii_stack_max_rows(int32_t f);
int dggb_gcnii_stack_fwd(const int32_t* rowptr, const int32_t* col, const float* val, int32_t n, const float* x0,
                         const float* h0, int32_t f, int32_t layers, const float* const* w_host_ptrs,
                         const float* theta_host, float c1, float c2, const float* keep, float* y, float* s_out,
                         uint32_t* barrier_zeroed, void* stream);

/* ------------------------------------------------------------------------------------
 * Node encoder forward: out[N,H] = LeakyReLU_slope(x[N,F] W[H,F]^T + b)  (slope = 1: plain Linear)
 * -- nn.Sequential(nn.Linear, nn.LeakyReLU) of dgm.py:1741-1744, 1097-1100, 1123-1126 and the
 * y = x_enc We^T product.  tcgen05 tensor cores with an in-kernel 3xTF32 split (fp32-level
 * accuracy, fp32 accumulate in TMEM): x tiles by TMA -> registers -> TMEM ("TS" MMA), W
 * pre-split into the workspace; x is read from HBM once.
 * Requires F % 4 == 0 and H in {16, 32, 64, 128} (else DGGB_ERR_BAD_SHAPE: use a library GEMM).
 * b may be NULL.
 * ---------------------------------------------------------------------------------- */
int64_t dggb_linear_act_workspace_bytes(int32_t f, int32_t h);   /* hi/lo split of W */
/* General form used by the fused encoder backward:
 *   v = x W_eff^T + b + addend;   out = act_src ? v * LeakyReLU'_slope(act_src) : LeakyReLU_slope(v)
 * W_eff = w ([H,F]) or, with w_transposed, w^T (w given as [F,H]).  With x = dy, w = We (transposed),
 * addend = dL/dx_enc, act_src = x_enc this is d pre = LeakyReLU'(x_enc) * (dy We + dL/dx_enc) in one pass
 * (autograd of dgm.py:1778-1784).  b / addend / act_src may be NULL.
 * w2/out2 (H in {32, 64}): additionally out2 = out w2^T, chained inside the same kernel (the activated tile
 * goes registers -> TMEM as the next A operand): x_enc and y = x_enc We^T of dgm.py:1778+1784 in one launch. */
int dggb_linear_fused(const float* x, const float* w, int32_t w_transposed, const float* b,
                      const float* addend /* [N,H] */, const float* act_src /* [N,H] */, float slope,
                      int32_t n, int32_t f, int32_t h, float* out,
                      const float* w2 /* [H,H] or NULL */, float* out2 /* [N,H] or NULL */,
                      void* workspace, int64_t workspace_bytes,
                      float* zero_ws /* or NULL: zero_count floats cleared before the GEMM starts (the
                                        split-K buffers of the weight gradients that follow) */,
                      int64_t zero_count,
                      void* splitk_ws /* or NULL: [splits, N, H] fp32 scratch of dggb_linear_splitk_workspace_bytes:
                                         few row tiles and a wide x (Cora / Citeseer raw features) are then split
                                         over k so that every SM streams; the partial tiles are summed in a fixed
                                         order by a second small launch (w2 == NULL only) */,
                      int64_t splitk_ws_bytes, void* stream);
int64_t dggb_linear_splitk_workspace_bytes(int32_t n, int32_t f, int32_t h);   /* 0: the call would not split */
int dggb_linear_act_fwd(const float* x, const float* w, const float* b, float slope, int32_t n,
                        int32_t f, int32_t h, float* out, void* workspace, int64_t workspace_bytes,
                        void* stream);
/* The node encoder + edge-encoder projection of class DGG as the training step runs them (dgm.py:1778, 1784 and
 * their autograd):
 *   dggb_encoder_fwd:  x_enc = LeakyReLU_slope(x Wn^T + bn),  y = x_enc We^T  (H in {32, 64}; == dggb_linear_fused with
 *     w2 = We).  Its weight-split launch additionally writes we_t_split [2H, H] = [We^T_hi ; We^T_lo] (or NULL) -- the
 *     pre-split B operand of the backward's d pre GEMM -- and clears zero_ws (the backward's accumulators), so the
 *     backward needs no split / fill launches of its own.
 *   dggb_encoder_bwd_dpre:  d pre = LeakyReLU'_slope(x_enc) * (g_y We + g_xenc)  (g_xenc may be NULL) in ONE launch.
 *     dpre [N,H] may be NULL when the caller only needs the weight gradients; dpre_t_hi / dpre_t_lo [H, npad]
 *     (npad >= n, npad % 4 == 0; both or neither) receive the TRANSPOSED TF32 hi/lo split of d pre, zero padded, and
 *     colsum[H] (or NULL) += its column sums (the bias gradient): the operands of dggb_gemm_tn_tc_presplit.
 *     gy_t_hi / gy_t_lo [H, npad] (both or neither): the same transposed split of the INPUT g_y, for the
 *     dWe = g_y^T x_enc product that dggb_gemm_tn_tc_presplit computes in the same launch as dWn = d pre^T x. */
int dggb_encoder_fwd(const float* x, const float* wn, const float* bn, float slope, int32_t n, int32_t f,
                     int32_t h, float* x_enc, const float* we, float* y, void* workspace,
                     int64_t workspace_bytes, float* we_t_split, float* zero_ws, int64_t zero_count,
                     void* stream);
int dggb_encoder_bwd_dpre(const float* g_y, const float* we_t_split, const float* g_xenc, const float* x_enc,
                          float slope, int32_t n, int32_t h, float* dpre, float* dpre_t_hi, float* dpre_t_lo,
                          int32_t npad, float* colsum, float* gy_t_hi, float* gy_t_lo, void* stream);

/* ------------------------------------------------------------------------------------
 * Weight gradients of the tall node encoders (nn.Linear of dgm.py:1741-1744 / 1097-1100 /
 * 1123-1126 applied to [N, F] features):  out[P,Q] += a[N,P]^T b[N,Q]  (dW = dpre^T x) and
 * colsum_a[P] += column sums of a (db); split over the N rows so every SM streams a slab.
 * out / colsum_a are ACCUMULATED INTO (zero them first); colsum_a may be NULL.  fp32 SIMT.
 * ---------------------------------------------------------------------------------- */
int dggb_gemm_tn_splitk(const float* a /* [N,P] */, const float* b /* [N,Q] */, int32_t n, int32_t p,
                        int32_t q, float* out /* [P,Q] */, float* colsum_a /* [P] or NULL */,
                        void* stream);
/* Same contract on the tcgen05 tensor cores (3xTF32 split in-kernel, b streamed by TMA once,
 * a transposed + split into the workspace).  Requires Q % 4 == 0, P in {16,32,64,128}. */
int64_t dggb_gemm_tn_tc_workspace_bytes(int32_t n, int32_t p);
int dggb_gemm_tn_tc(const float* a, const float* b, int32_t n, int32_t p, int32_t q, float* out,
                    float* colsum_a, void* workspace, int64_t workspace_bytes, void* stream);
/* Same product from an operand that is already transposed and split (a_t_hi / a_t_lo [P, npad], zero padded for
 * nodes >= n; written by dggb_encoder_bwd_dpre): no transpose pass, no workspace.  a2_t_hi / a2_t_lo / b2 [N, q2] /
 * out2 [P, q2] (all or none; q2 <= 128): a second, narrow product out2 += a2^T b2 over the same nodes computed by
 * extra CTAs of the same launch (dWe = g_y^T x_enc next to dWn = d pre^T x). */
int dggb_gemm_tn_tc_presplit(const float* a_t_hi, const float* a_t_lo, int32_t npad, const float* b, int32_t n,
                             int32_t p, int32_t q, float* out, const float* a2_t_hi, const float* a2_t_lo,
                             const float* b2, int32_t q2, float* out2, void* stream);

/* ------------------------------------------------------------------------------------
 * All-pairs scoring + per-row streaming top-K (legacy all-pairs DGG, dgm.py:271-301; a15):
 *
 *   y_ij = -t * || z_i - z_j ||_2  [+ noise_ij]          (cdist -> exp -> log -> + Gumbel)
 *   per query row: the Kc largest y_ij, sorted descending (ties: lower column first), i.e.
 *   the first Kc columns of torch.sort(y, descending=True) -- the only ones the soft first-k
 *   curve leaves non-zero (SURVEY.md section 0).
 *
 * Z Z^T runs on the tcgen05 tensor cores (kind::tf32; precision = 3: 3xTF32 split, ~fp32
 * accuracy; precision = 1: single TF32 pass), operands staged by TMA, accumulators in TMEM;
 * the epilogue fuses norms, sqrt, temperature, noise and the selection.  No N x N matrix is
 * written.  Rows [row_begin, row_begin+row_count) are scored against all n columns (row
 * sharding across GPUs: every rank passes the all-gathered z and its own row block).
 *   noise: [row_count, noise_ld] fp32 (row r of it belongs to query row row_begin+r) for parity
 *          runs with an injected tensor; or NULL, in which case noise_scale != 0 selects
 *          counter-based Gumbel(0, noise_scale) noise generated in the epilogue: Philox4x32-7,
 *          key = seed, counter = (global row, col >> 2), output lane col & 3; the same (row, col)
 *          always regenerates the same value, so shards and recomputation agree without
 *          communication (tests/philox_ref.py is the host restatement).
 *   out_idx/out_val: [row_count, kc]; unused slots (n < kc) hold idx -1 / val 0.
 *   workspace: dggb_allpairs_workspace_bytes(n, d) bytes (hi/lo split of z + squared norms).
 *   out_rowsum (optional): sum_j exp(y_ij * inv_temp) over ALL n columns -- the normaliser of the
 *          evaluation branch softmax(log_p / temp) (dgm.py:298), accumulated in the same pass.
 * Requires kc <= 64; any d.  For d > 128 (d rounded up to 32) a k-block-streamed kernel runs the call: the query
 *   tile is streamed 32 features at a time with each key tile, so shared memory does not depend on d.  It runs
 *   unsplit; DGGB_AP_V1 and DGGB_AP_PARTS have no effect on it.
 *   Column parts: when the row blocks of a call fill the SMs badly (a row-sharded rank: 228 blocks on 148 SMs), the
 *   column range is cut into up to 8 parts scored by separate CTAs and a merge launch picks the best kc of a row's
 *   parts (same order, identical result).  That needs parts * row_count * kc * 8 more workspace bytes:
 *   dggb_allpairs_workspace_bytes_rows() returns the size including them; with only the base size the call runs unsplit.
 *   DGGB_AP_PARTS=1..8 overrides the choice.
 * ---------------------------------------------------------------------------------- */
int64_t dggb_allpairs_workspace_bytes(int32_t n, int32_t d);
int64_t dggb_allpairs_workspace_bytes_rows(int32_t n, int32_t d, int32_t row_count, int32_t kc);
int dggb_allpairs_topk_fwd(const float* z /* [n,d] */, int32_t n, int32_t d, int32_t row_begin,
                           int32_t row_count, const float* t /* [1] device */, const float* noise,
                           int64_t noise_ld, uint64_t seed, float noise_scale, int32_t kc,
                           int32_t precision, void* workspace,
                           int64_t workspace_bytes, int32_t* out_idx, float* out_val, float inv_temp,
                           float* out_rowsum /* [row_count] or NULL */, void* stream);
/* Continuation pass for rows that need more than 64 selected entries (k_i unbounded above, SURVEY 7.3): as
 * dggb_allpairs_topk_fwd, but only entries that sort strictly AFTER (after_val[r], after_idx[r]) -- the last entry
 * the previous pass returned for row r -- in (value descending, column ascending) order are admitted; pass p + 1 of
 * a row therefore returns ranks [64 p, 64 (p + 1)).  after_val / after_idx: [row_count], both or neither NULL.
 * A row whose after_idx is -1 (the previous pass ran out of columns) admits nothing: all its slots come back empty. */
int dggb_allpairs_topk_after_fwd(const float* z, int32_t n, int32_t d, int32_t row_begin, int32_t row_count,
                                 const float* t, const float* noise, int64_t noise_ld, uint64_t seed,
                                 float noise_scale, int32_t kc, int32_t precision, void* workspace,
                                 int64_t workspace_bytes, const float* after_val, const int32_t* after_idx,
                                 int32_t* out_idx, float* out_val, float inv_temp, float* out_rowsum,
                                 void* stream);
/* Backward by recomputation over the selected pairs only (O(rows*kc*d)):
 * dz[n,d] and dt[1] are ACCUMULATED INTO. */
int dggb_allpairs_pair_bwd(const float* z, int32_t n, int32_t d, int32_t row_begin, int32_t row_count,
                           const int32_t* idx, const float* gy /* [row_count,kc] */, int32_t kc,
                           const float* t, float* dz, float* dt, void* stream);

/* ------------------------------------------------------------------------------------
 * One-shot all-reduce (sum) of a flat fp32 buffer over NVLink peer memory, for use INSIDE a captured step: the
 * data-parallel drivers sum the replicated DGG / conv weight gradients after every backward (SURVEY 8e); as an NCCL
 * call that is a fixed 20-35 us launch behind a ~110 us step.
 *   bufs_dev  [world] device array: pointer to every rank's symmetric buffer (peer-mapped; index = rank)
 *   pads_dev  [world] device array: pointer to every rank's signal pad (uint32 slots, zero on first use); slots
 *             [pad_slot_base, pad_slot_base + 2 world) are used
 *   out       [count] local result (may not alias the symmetric buffer: peers read it until the end barrier)
 *   state     [2] uint32, zero on first use: sequence number + block counter (device-resident: graph replays
 *             cannot change kernel arguments)
 *   multicast_ptr: NULL, or the NVSwitch multicast address of the same buffers -- then ONE multimem.ld_reduce per
 *             16 bytes replaces the `world` peer loads (the switch does the sum)
 * Every rank must call it the same number of times; count % 4 == 0; world <= 16.
 * ---------------------------------------------------------------------------------- */
int dggb_allreduce_oneshot(void* const* bufs_dev, void* const* pads_dev, int32_t rank, int32_t world, int64_t count,
                           float* out, uint32_t* state, const void* multicast_ptr, int32_t pad_slot_base,
                           int32_t blocks, int32_t end_barrier /* 0: the caller alternates two buffers */,
                           void* stream);

/* ------------------------------------------------------------------------------------
 * Sub-graph sampling on the device (SURVEY 8f rank 2): what torch_geometric.loader.GraphSAINTRandomWalkSampler does
 * for train_large_graphs.py:402-413 / train_reddit.py:400-411 (third-party, not in the reference tree: semantics of
 * torch_sparse random_walk + saint_subgraph restated; parity unpinned, see DESIGN.md).
 *   dggb_random_walk: walk[w][0] = start[w]; step s moves to entry floor(u * deg) of the current row's CSR range,
 *     u = (x >> 8) / 2^24 with x = 32-bit lane (s & 3) of Philox4x32-7(counter = (walker_offset + w, s >> 2), key = seed);
 *     a node without out-edges keeps the walker in place.  walk is [num_walkers, walk_length + 1] int32.
 *   dggb_induced_subgraph_count / _fill: the sub-graph induced by the SORTED, unique node list nodes[m]:
 *     count fills relabel[n] (position in nodes, or -1) and counts[m + 1] (kept entries per selected row, counts[m] = 0);
 *     the caller scans counts into sub_rowptr[m + 1]; fill writes the kept entries in row-major order:
 *     sub_col (relabelled column) and sub_eid (position of the entry in the parent CSR).
 * ---------------------------------------------------------------------------------- */
int dggb_random_walk(const int32_t* rowptr, const int32_t* col, int32_t n, const int32_t* start,
                     int32_t num_walkers, int32_t walk_length, uint64_t seed, int64_t walker_offset, int32_t* walk,
                     void* stream);
int dggb_induced_subgraph_count(const int32_t* rowptr, const int32_t* col, int32_t n, const int32_t* nodes, int32_t m,
                                int32_t* relabel, int32_t* counts, void* stream);
int dggb_induced_subgraph_fill(const int32_t* rowptr, const int32_t* col, const int32_t* nodes, int32_t m,
                               const int32_t* relabel, const int32_t* sub_rowptr, int32_t* sub_col, int32_t* sub_eid,
                               void* stream);

/* ------------------------------------------------------------------------------------
 * k-hop neighbour sampling on the device: what torch_geometric.loader.NeighborLoader (torch_sparse / pyg-lib
 * neighbor_sample, third-party, not in the reference tree) does for train_pubmed.py:370-375.  Parity with PyG is
 * unpinned: the RNG stream differs and so does the within-target order of Floyd's picks; tests/neighbor_ref.py
 * restates the contract below as a sequential loop and the kernels match it bit for bit.
 *
 * The parent graph is in CSC form, colptr[n+1] / row[nnz]: the entries of target v are its in-neighbours (sources u
 * of the edges u -> v) sorted by source; multi-edges stay separate entries.  Hop l (0-based, l < 255) has frontier F_l
 * and fanout k_l: F_0 = the seeds, F_{l+1} = the nodes first discovered in hop l, in discovery order.  For frontier
 * slot t (position in F_l) with target v and d = deg_in(v):
 *   - d == 0 or k == 0: nothing;
 *   - k < 0, or replace == 0 and k >= d: all d entries in ascending position;
 *   - replace == 1: k draws, draw i emits position floor(x_i * d / 2^32), in draw order;
 *   - otherwise Floyd's algorithm (as torch_sparse): for i = 0..k-1, j = d - k + i, r = floor(x_i * (j+1) / 2^32);
 *     add r to the set, or j if r is already in it; the k positions are emitted in ascending order.
 *   x_i = 32-bit lane (i & 3) of Philox4x32-7(counter = (t, (l << 24) | (i >> 2)), key = seed) (csrc/philox.cuh).
 *   k <= 1024 (larger: DGGB_ERR_BAD_SHAPE); k = -1 means "all".
 * Emissions of a hop are ordered by slot, then by the per-target order above.  A source not yet in n_id gets the next
 * local id at its first emission (torch_sparse's sequential rule); every emission is one edge (local(u), local(v)).
 *
 * Workspace: local[n] (local id or -1) and claim[n] (INT_MAX when idle), filled once by the caller; a batch leaves
 * them as it found them once dggb_neighbor_reset has run over its n_id.  Per batch:
 *   dggb_neighbor_seed: local[seeds[t]] = t; *status = 1 if a seed is out of range or repeated, else 0.
 * Per hop (frontier[m], the local id of slot t is frontier_base + t):
 *   dggb_neighbor_count: counts[m] int64 emissions per slot; the caller scans them (int64, inclusive) into offsets
 *     and reads the total T, which must be <= 2^31 - 1;
 *   dggb_neighbor_sample: out_pos[T] (CSC positions), out_dst[T] (target local ids), and claim[u] = the smallest
 *     emission index of every source u with local[u] < 0;
 *   dggb_neighbor_flag: flags[T] = 1 at the first emission of each new source; the caller scans them (int32,
 *     inclusive) into scan and reads the number of new nodes;
 *   dggb_neighbor_assign: new_nodes[id] = u and local[u] = base + id, id = scan[e] - 1 at each flagged emission.
 * Once the last hop is assigned:
 *   dggb_neighbor_edges: edge_index[2, count] int64 = (local source, dst) of every emission (hops concatenated);
 *   dggb_neighbor_reset: local[u] = -1, claim[u] = INT_MAX for the nodes[count] of the batch.
 * ---------------------------------------------------------------------------------- */
int dggb_neighbor_seed(const int32_t* seeds, int32_t num_seeds, int32_t n, int32_t* local, int64_t* status,
                       void* stream);
int dggb_neighbor_count(const int32_t* colptr, int32_t n, const int32_t* frontier, int32_t m, int32_t k,
                        int32_t replace, int64_t* counts, void* stream);
int dggb_neighbor_sample(const int32_t* colptr, const int32_t* row, const int32_t* frontier, int32_t m, int32_t k,
                         int32_t replace, int32_t hop, uint64_t seed, int32_t frontier_base, const int64_t* offsets,
                         const int32_t* local, int32_t* claim, int32_t* out_pos, int32_t* out_dst, void* stream);
int dggb_neighbor_flag(const int32_t* row, const int32_t* pos, int32_t count, const int32_t* local,
                       const int32_t* claim, int32_t* flags, void* stream);
int dggb_neighbor_assign(const int32_t* row, const int32_t* pos, int32_t count, const int32_t* flags,
                         const int32_t* scan, int32_t base, int32_t* local, int32_t* new_nodes, void* stream);
int dggb_neighbor_edges(const int32_t* row, const int32_t* pos, const int32_t* dst, int64_t count,
                        const int32_t* local, int64_t* edge_index, void* stream);
int dggb_neighbor_reset(const int32_t* nodes, int32_t count, int32_t n, int32_t* local, int32_t* claim,
                        void* stream);

/* ------------------------------------------------------------------------------------
 * Deterministic multilevel k-way graph partitioning on the device: what METIS does for torch_geometric.loader.ClusterData
 * (train_large_graphs.py:402-421; third-party, host cores).  The partitions are NOT METIS's: parity is unpinned;
 * tests/cluster_ref.py restates every phase below and the driver of dgg_b200.samplers.partition, and the kernels match
 * it bit for bit.  Integer arithmetic only; atomics compute only sums and minima, so no result depends on the order in
 * which blocks or atomics run.
 *
 * A level is a symmetric CSR rowptr[n+1] / col[nnz] (rows sorted, no self loops, no duplicates) with entry weights
 * ewt[nnz] >= 1 and node weights vw[n] >= 1.  A labelling lab[n] assigns every node a label (a cluster while
 * coarsening, a part while refining) in [0, nlabels).  h(x) = MurmurHash3's fmix32.  NONE = INT64_MAX.
 *   dggb_partition_weights: lw[L] = sum of vw over the nodes labelled L; anchor[L] = the smallest such node, or
 *     0x7f7f7f7f (anchor may be NULL).
 *   dggb_partition_propose: key[n].  Each active node v finds the adjacent label L != lab[v] with
 *     lw[L] + vw[v] <= limit that has the largest (conn(L), h(L)), conn(L) = summed ewt of v's entries into L, and
 *     gain = conn(L) - conn(lab[v]).  mode 0 (cluster): active when (h(v) & 1) == parity; proposes L when gain > 0.
 *     mode 1 (refine): as 0, and v != anchor[lab[v]] (a part is never left empty).  mode 3 (unload): as 1, and
 *     lw[lab[v]] > limit; proposes L whatever the gain.  A proposal is key = L << 32 | (uint32)(2^31 - 1 - gain), no
 *     proposal NONE.  mode 2 (evict): every v != anchor[lab[v]] with lw[lab[v]] > limit (parity ignored) gets
 *     key = lab[v] << 32 | (uint32)(2^31 - 1 - gain), conn(L) = 0 when there is no L.  anchor may be NULL in mode 0.
 *   The caller sorts the keys stably (node id breaks ties) into keys[n] / order[n] (int64).
 *   dggb_partition_admit: cum[n] = inclusive int64 scan of vw[order].  Each run of equal target t = key >> 32 is
 *     admitted in order while lw[t] (start-of-round weight) + the run's weight up to and including the node <= limit:
 *     lab[order[i]] = t.
 *   dggb_partition_rebalance (unit node weights): for the evict keys of mode 2 with limit = cap, the first
 *     lw[p] - cap nodes of each over-full part p (least gain lost first) take the free places cap - lw[q] of the parts
 *     below cap in part order: ex_prefix[k] = exclusive scan of max(lw - cap, 0), room_cum[k] = inclusive scan of
 *     max(cap - lw, 0), both int64.
 *   dggb_partition_contract_keys: keys[nnz] = cluster[row] * nc + cluster[col] of every entry, NONE inside a cluster.
 *     The caller sorts them (any sort: idx[nnz] = the source entry of each sorted key).
 *   dggb_partition_contract_heads: heads[nnz] int32 = 1 at the first of each run of equal sorted keys (not NONE); the
 *     caller scans them (int32, inclusive) into scan and reads cnnz = scan[nnz-1].
 *   dggb_partition_contract_fill: coarse entry j = scan - 1 of a run: crow[j] (int64), ccol[j], cwt[j] = summed ewt[idx].
 *   dggb_partition_bfs: order[n], pos[n] (position in order) of a level-synchronous BFS: a frontier node's unvisited
 *     neighbours follow it ordered by (parent position, id); a new search starts from the smallest unvisited id.
 *     claim[n] is scratch.  One block: meant for the coarsest level.
 *   dggb_partition_chunk: part[order[i]] = min(k - 1, prefix[i] * k / total), prefix = exclusive int64 scan of
 *     vw[order], total = its sum.
 *   dggb_partition_project: out[v] = map[idx[v]].
 * ClusterLoader batches over the parent CSR permuted so that every part is a contiguous id range:
 *   dggb_cluster_batch_count / _fill: drawn part b covers parent ids [start[b], end[b]) and local ids from base[b];
 *     rows node_idx[m] are the drawn parts' ids in draw order.  count: counts[m] kept entries per row (columns inside
 *     a drawn part); the caller scans them into sub_rowptr[m + 1].  fill: each row's kept entries in ascending local
 *     id, i.e. one ascending run per drawn part in draw order: sub_col (local id), sub_eid (position in the parent CSR).
 * ---------------------------------------------------------------------------------- */
int dggb_partition_weights(const int32_t* lab, const int32_t* vw, int32_t n, int32_t nlabels, int32_t* lw,
                           int32_t* anchor, void* stream);
int dggb_partition_propose(const int32_t* rowptr, const int32_t* col, const int32_t* ewt, const int32_t* vw,
                           const int32_t* lab, int32_t n, const int32_t* lw, const int32_t* anchor, int32_t limit,
                           int32_t parity, int32_t mode, int64_t* key, void* stream);
int dggb_partition_admit(const int64_t* keys, const int64_t* order, const int64_t* cum, int32_t n, const int32_t* lw,
                         int32_t limit, int32_t* lab, void* stream);
int dggb_partition_rebalance(const int64_t* keys, const int64_t* order, int32_t n, const int32_t* lw,
                             const int64_t* ex_prefix, const int64_t* room_cum, int32_t k, int32_t cap, int32_t* part,
                             void* stream);
int dggb_partition_contract_keys(const int32_t* rowptr, const int32_t* col, int32_t n, const int32_t* cluster,
                                 int32_t nc, int64_t* keys, void* stream);
int dggb_partition_contract_heads(const int64_t* keys, int64_t nnz, int32_t* heads, void* stream);
int dggb_partition_contract_fill(const int64_t* keys, const int64_t* idx, const int32_t* ewt, int64_t nnz,
                                 const int32_t* scan, int32_t nc, int32_t cnnz, int64_t* crow, int32_t* ccol,
                                 int32_t* cwt, void* stream);
int dggb_partition_bfs(const int32_t* rowptr, const int32_t* col, int32_t n, int32_t* order, int32_t* pos,
                       int32_t* claim, void* stream);
int dggb_partition_chunk(const int32_t* order, const int64_t* prefix, int32_t n, int64_t total, int32_t k,
                         int32_t* part, void* stream);
int dggb_partition_project(const int32_t* map, const int32_t* idx, int32_t n, int32_t* out, void* stream);
int dggb_cluster_batch_count(const int32_t* rowptr, const int32_t* col, const int32_t* start, const int32_t* end,
                             int32_t num_drawn, const int32_t* node_idx, int32_t m, int32_t* counts, void* stream);
int dggb_cluster_batch_fill(const int32_t* rowptr, const int32_t* col, const int32_t* start, const int32_t* end,
                            const int32_t* base, int32_t num_drawn, const int32_t* node_idx, int32_t m,
                            const int32_t* sub_rowptr, int32_t* sub_col, int32_t* sub_eid, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DGGB_H_ */
