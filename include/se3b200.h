/* se3b200.h -- C ABI of the B200-native SE(3)-Transformer attention hot path.
 *
 * The reference (lucidrains/se3-transformer-pytorch @ e1669ee) has no FFI layer: its boundary is the
 * Python class SE3Transformer.  This header declares the entry points a native replacement of the hot
 * path binds at the three tensor-only seams of the reference (SURVEY.md section 8b):
 *
 *   neighbour builder inside SE3Transformer.forward   se3_transformer_pytorch.py:1171-1294  -> se3_knn_fwd
 *   get_basis(r_ij, max_degree)                        basis.py:153-205                      -> se3_basis_fwd
 *   RadialFunc trunk (net.0 .. net.5)                  se3_transformer_pytorch.py:287-293    -> se3_radial_trunk_fwd
 *   PairwiseConv + ConvSE3 inner product               se3_transformer_pytorch.py:237-254,
 *                                                      326-343                               -> se3_tbuild_fwd +
 *                                                                                               se3_pairwise_{simt,tc}_fwd
 *   masked_mean pooling of ConvSE3                     utils.py:72-80, S:256-257             -> se3_pool_fwd
 *   AttentionSE3.forward logits/softmax/aggregate      se3_transformer_pytorch.py:476-517    -> se3_attn_fwd
 *     (low-rank radial path: se3_pack_lowrank + se3_pairwise_lr_fwd, se3_fold_basis_fwd, se3_rotate_back_fwd:
 *      the same product re-associated; DESIGN.md 4.2-4.4)
 *   NormSE3.forward (next to the hot path, SURVEY 8f)  se3_transformer_pytorch.py:130-152    -> se3_norm_fwd
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to a contiguous row-major buffer unless marked HOST;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing synchronises;
 *   - buffers are borrowed for the duration of the call; the library keeps no state between calls;
 *   - return value 0 = success; otherwise a negative SE3_E* code and se3_last_error() (HOST string,
 *     thread-local) describes the failure.  No CPU fallback exists.
 *   - fp32 arithmetic throughout; the tensor-core kernel evaluates its one dense contraction as a
 *     3-pass fp16 split (x = hi + lo, 22 mantissa bits; hi*hi + lo*hi + hi*lo, fp32 accumulate), error < 1e-6 relative.
 */
#ifndef SE3B200_H
#define SE3B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SE3_OK            0
#define SE3_EINVAL       -1   /* bad argument / unsupported shape */
#define SE3_ECUDA        -2   /* CUDA runtime error (launch, attribute) */
#define SE3_RADIAL_MID   128  /* RadialFunc mid_dim, se3_transformer_pytorch.py:278 */
#define SE3_TILE_E       128  /* edges per tile (UMMA M) */
#define SE3_TILE_O        32  /* output channels per tile */
#define SE3_TILE_IF        4  /* (in-channel, frequency) pairs per tile step */

const char* se3_last_error(void);
int         se3_abi_version(void);

/* Neighbour graph (S:1171-1294).  For every node i of every cloud: the k smallest "modified" distances over the
 * other n-1 nodes, ascending (ties: lower node index first), exactly as the reference's remove-self + topk:
 *   modified = true distance; user neighbor_mask==0 -> FLT_MAX (S:1257); bonded (sparse_adj!=0) -> 0 (S:1262);
 *   causal and j' >= i on the self-removed grid -> FLT_MAX (S:1266-1268).
 * out_mask = (modified <= valid_radius) & node_mask[i] & node_mask[j]  (S:1284, 1290-1291).
 * node_mask, neighbor_mask, sparse_adj may be NULL.  Requires 1 <= k <= n-1 and n-1 <= 4096. */
int se3_knn_fwd(const float* coors, const uint8_t* node_mask, const uint8_t* neighbor_mask, const uint8_t* sparse_adj,
                int b, int n, int k, float valid_radius, int causal,
                int64_t* out_idx, uint8_t* out_mask, float* out_rel_pos, float* out_rel_dist, void* stream);

/* Gather per-pair features onto the neighbour list (batched_index_select at S:1293-1294, utils.py:56-70):
 * out[b,i,kk,:] = pair_feat[b,i,idx[b,i,kk],:]   with pair_feat [b,n,n,e]. */
int se3_gather_pairs_fwd(const float* pair_feat, const int64_t* idx, int b, int n, int k, int e, float* out, void* stream);

/* Equivariant basis (basis.py:153-205): real spherical harmonics Y_J, J <= 2*max_degree, evaluated from Cartesian
 * r_ij without trigonometry, times the constant Q_J tables given as a CSR matrix over R = sum_pairs (2lo+1)(2li+1)f rows
 * and sum_J (2J+1) columns.  Pair p occupies out[pair_base[p]*E .. ) as [E, rows_p] row-major, rows_p =
 * pair_row0[p+1]-pair_row0[p]; within a pair row = (p_out*(2li+1)+q_in)*f + f_idx (B:197-198). */
int se3_basis_fwd(const float* rel_pos, int64_t E, int max_degree,
                  const int32_t* csr_row_ptr, const int32_t* csr_col, const float* csr_val,
                  const int32_t* pair_row0, const int32_t* pair_base, int num_pairs,
                  float* out, void* stream);

/* Radial trunk (S:287-293) for `num_pairs` independent RadialFunc MLPs over the same edge features:
 * g = GELU(LN(W2 GELU(LN(W1 feat + b1)) + b2)), exact erf GELU, LN eps 1e-5.
 * params: per pair, contiguous floats [W1^T (in_dim x 128) | b1 | ln1_w | ln1_b | W2^T (128 x 128) | b2 | ln2_w | ln2_b].
 * out_g: [num_pairs, E, 128] fp32. */
int se3_radial_trunk_fwd(const float* feat, int64_t E, int in_dim, int num_pairs, const float* params,
                         float* out_g, void* stream);

/* T[e,i,f,p] = sum_q basis[e,p,q,f] * x[b, idx[e], i, q]   (the gather at S:237 fused with the basis contraction of
 * the factored form, SURVEY.md A.4).  x: [b,n,Ci,Q], basis_pair: [E,P,Q,F], E = b*n*k.  Edge tiles
 * [tile_begin, tile_begin+tile_count) (128 edges each) are written to T in tile layout
 * [tile_count][ceil(Ci*F/4)][4][ceil(P/4)][128][4] floats (zero padded), so a ConvSE3 can be evaluated in edge chunks
 * (the B200 counterpart of the reference's node-axis `splits`, S:243-252). */
int se3_tbuild_fwd(const float* x, const int64_t* idx, const float* basis_pair, int b, int n, int k,
                   int Ci, int P, int Q, int F, int64_t tile_begin, int64_t tile_count, float* T, void* stream);

/* out[e,o,p] (+)= sum_{i,f} (W3[(o*Ci+i)*F+f,:].g[e,:] + b3[(o*Ci+i)*F+f]) * T[e,i,f,p]     (S:299, 336-343, 251-254)
 * fp32 SIMT version, any shape.  g: [E,128]; W3: [Co*Ci*F,128]; out: [E,Co,P]. */
int se3_pairwise_simt_fwd(const float* g, const float* W3, const float* b3, const float* T,
                          int64_t E, int Co, int Ci, int F, int P, int accumulate, float* out, void* stream);

/* Pack RadialFunc.net.6 weight/bias into the tensor-core operand image (once per weight update).
 * bytes needed: se3_w3_image_bytes(Co, Ci, F).  Requires Co % 32 == 0 and |W3| < 6e4 (fp16 hi/lo split). */
int64_t se3_w3_image_bytes(int Co, int Ci, int F);
int se3_pack_w3(const float* W3, const float* b3, int Co, int Ci, int F, void* image, void* stream);

/* Same contraction as se3_pairwise_simt_fwd on the tcgen05 tensor cores (sm_100a only): g [E,128] fp32 from
 * se3_radial_trunk_fwd (one pair's slice; split to fp16 hi/lo into tensor memory inside the kernel), w_img from
 * se3_pack_w3, T from se3_tbuild_fwd. */
int se3_pairwise_tc_fwd(const float* g, const void* w_img, const float* T,
                        int64_t E, int Co, int Ci, int F, int P, int accumulate, float* out, void* stream);
/* Diagnostic for tests: as above, and dumps (R + bias) of the first (i,f) step as [ceil(E/128), Co/32, 128, 128] fp32
 * (column = if_local*32 + o_local). */
int se3_pairwise_tc_debug(const float* g, const void* w_img, const float* T, int64_t E, int Co, int Ci, int F,
                          int P, int accumulate, float* out, float* dumpR, void* stream);

/* Low-rank radial path.  When the trunk outputs of a pair, G [E,128], factor as G ~= U V^T with small rank r (distance-only
 * radial functions: r ~ 16, see DESIGN.md section 4.2), the host passes
 *   U  [E, 64] fp32: columns 0..r-1 = G V, column r = 1 (bias slot), remaining columns 0;
 *   Fp [Co*Ci*F, Kp] fp32: columns 0..r-1 = W3 V, column r = b3, remaining 0;  Kp = 16*ceil((r+1)/16) <= 64
 * se3_pack_lowrank images Fp for the tensor cores (se3_lowrank_image_bytes bytes) and se3_pairwise_lr_fwd evaluates the
 * same contraction as se3_pairwise_tc_fwd with K = Kp instead of 128 (bias folded into the GEMM). */
int64_t se3_lowrank_image_bytes(int Co, int Ci, int F, int Kp);
int se3_pack_lowrank(const float* Fp, int Co, int Ci, int F, int Kp, void* image, void* stream);
int se3_pairwise_lr_fwd(const float* U, const void* w_img, const float* T, int64_t E, int Co, int Ci, int F, int P,
                        int Kp, int accumulate, float* out, void* stream);

/* Basis fold of the input-side contraction (pairs with 2 l_in + 1 = Q < P = 2 l_out + 1; S:336-343, 251 reassociated):
 *   out[e,o,p] (+)= sum_{f,q} basis_pair[e,p,q,f] * S[f,e,o,q]
 * where S[f] [E,Co,Q] = se3_pairwise_lr_fwd with F := 1, P := Q, T := the gathered neighbour features in tile layout
 * (se3_tbuild_fwd with an identity basis) and the image of frequency f's rows of Fp.  basis_pair: [E,P,Q,F] of these E edges. */
int se3_fold_basis_fwd(const float* S, const float* basis_pair, int64_t E, int Co, int P, int Q, int F, int accumulate,
                       float* out, void* stream);
/* Rotation of the edge-aligned outputs back to the global frame (DESIGN.md 4.4): out[e,o,:] = D_lo(e) out'[e,o,:], D [E,P,P],
 * out' given as one dense buffer per |m|: part0 [E,Co] (m = 0), part_m [E,Co,2] = components (+m, -m); NULL = zero. */
int se3_rotate_back_fwd(const float* part0, const float* part1, const float* part2, const float* part3, const float* D,
                        int64_t E, int Co, int lo, float* out, void* stream);
/* Same fold with S stored component-major, S[f,e,q,o] ([F,E,Q,Co]): the rotation of the edge-aligned outputs back to the
 * global frame, out[e,o,:] = D_lo(e) out'[e,:,o]  (F = 1, Q = P, basis_pair = D_lo). */
int se3_fold_basis_cm_fwd(const float* S, const float* basis_pair, int64_t E, int Co, int P, int Q, int F, int accumulate,
                          float* out, void* stream);

/* Diagnostic for tools/: as se3_pairwise_lr_fwd; CTA 0 writes clock64 stamps of its warp roles to trace[5][64][8] (u64). */
int se3_pairwise_lr_trace(const float* U, const void* w_img, const float* T, int64_t E, int Co, int Ci, int F, int P,
                          int Kp, int accumulate, float* out, unsigned long long* trace, void* stream);

/* ---- production path of distance-only radial functions: low-rank radial basis + edge-aligned frames as one GEMM per
 * (degree_out, |m|) (DESIGN.md 4.5; the same product S:237-254, 326-343 re-associated) ------------------------------------ */

/* Radial trunk as se3_radial_trunk_fwd, followed in the same kernel by the low-rank radial coordinates of every pair:
 *   out_U [num_pairs, E, 64]: columns 0..r-1 = (g - gmean) V, column r = 1 (bias slot), rest 0, r = ones_col[pair],
 *   V [num_pairs,128,64] (columns >= r zero), gmean [num_pairs,128] the centre of the pair's radial curve (W3 gmean is part of the
 *   bias column of F');  stats [num_pairs, 2] (caller zeroes it): (max |g - gmean - U V^T|, max |g|) over the edges, accumulated with
 *   atomicMax -- the run-time check that the cached basis covers this forward's distances, read by the host once per forward.
 *   out_g may be NULL. */
int se3_radial_trunk_u_fwd(const float* feat, int64_t E, int in_dim, int num_pairs, const float* params, const float* V,
                           const float* gmean, const int* ones_col, float* out_g, float* out_U, float* stats, void* stream);

/* Radial coordinates by table lookup (distance-only radial functions): out_U as se3_radial_trunk_u_fwd, interpolated (4-point
 * Lagrange) from table [num_pairs, G, KT] fp32 = U(d) sampled on the uniform grid d_i = i Dmax / (G - 1) (built in float64 with
 * the plan; columns >= r zero), dist [E] the neighbour distances.  A distance outside [0, Dmax] (or NaN) sets stats[pair] = (1, 1):
 * the plan does not cover this forward. */
int se3_radial_table_fwd(const float* dist, int64_t E, const float* table, int G, int KT, float Dmax, const int* ones_col,
                         int num_pairs, float* out_U, float* stats, void* stream);

/* Per-edge frames: R_e takes the polar axis a = (0,1,0) of the reference's harmonics (basis.py:57-95) to the direction of
 * rel_pos[e]; D_out[l] [E, 2l+1, 2l+1] = real Wigner matrix D_l(R_e) in the reference's basis, l = 1..lmax <= 5, computed in
 * float64 as Y_l(R x_s) pinv(Y_l(x_s)) from the tables xs[l] [n_samples[l], 3] / pin[l] [2l+1, n_samples[l]] (device, float64).
 * xs, pin, n_samples, D_out: HOST arrays indexed by l (entry 0 unused). */
int se3_frames_fwd(const float* rel_pos, int64_t E, int lmax, const double* const* xs, const double* const* pin,
                   const int* n_samples, float* const* D_out, void* stream);

/* Neighbour gather (S:237-238, utils.py:56-70) fused with the rotation into the edge frame:
 *   X[tile][i][n][edge_local] = sum_q D[e][q][n] * x[b, idx[e], i, q],   x [b,n,Ci,Q], D [E,Q,Q] (NULL for Q = 1),
 * for the edge tiles [tile_begin, tile_begin + tile_count) of 128 edges (rows past E are zero). */
int se3_rotgather_fwd(const float* x, const int64_t* idx, const float* D, int b, int n, int k, int Ci, int Q,
                      int64_t tile_begin, int64_t tile_count, float* X, void* stream);

/* Pooled ConvSE3 epilogue (S:256-266, utils.py:72-80) fused with the rotation back to the global frame:
 *   out[node,o,:] = masked_mean_j( D_lo(e_j) Oprime[e_j,:,o] ) + self_add[node,o,:],   e_j = node*K + j,
 * Oprime [nodes*K, 2lo+1, Co] (component-major rows from se3_zgemm_fwd), D [nodes*K, 2lo+1, 2lo+1] (NULL for lo = 0),
 * mask [nodes*K] or NULL (plain mean), self_add [nodes, Co, 2lo+1] or NULL (the LinearSE3 self-interaction), out [nodes, Co, 2lo+1]. */
int se3_rotate_pool_fwd(const float* Oprime, const float* D, const uint8_t* mask, const float* self_add, int64_t nodes, int K,
                        int Co, int lo, float* out, void* stream);

/* out[row] = max_c |x[row, c]| (combine != 0: max with the value already in out); x [rows, W]. */
int se3_rowabsmax_fwd(const float* x, int64_t rows, int W, int combine, float* out, void* stream);
/* sx[e] = power of two with nodemax[b(e), idx[e]] * sqrt(2 max_degree + 1) * sx[e] < 2^10 (1 for all-zero nodes). */
int se3_edge_scale_fwd(const float* nodemax, const int64_t* idx, int b, int n, int k, int max_degree, float* sx, void* stream);

/* One K segment of se3_zgemm_fwd: radial coordinates U (row stride 64 floats; the segment uses the 16 columns at the pointer),
 * rotated neighbour features X from se3_rotgather_fwd ([tiles][Ci][ncomp][128]) and the component indices read from it. */
typedef struct se3_zseg {
  const float* U;
  const float* X;
  int Ci, ncomp, cplus, cminus;
} se3_zseg;

/* out'[e, plane c, o] = sum over segments, i, f, k of  Z_c[e,(seg,i,f,k)] * F'[o,(seg,i,f,k)]   with
 *   mode 1 (|m| = 0):  Z = U[e,k] x'[e,i,cplus]                                    (one plane, F = 1)
 *   mode 2 (|m| > 0):  Z_+ = (f=a: U x'[cplus], f=b: -U x'[cminus]),  Z_- = (f=a: U x'[cminus], f=b: U x'[cplus])   (two planes)
 *   mode 3 (|m| > 0):  the same two planes with three real products per complex one (Gauss): S1 = sum (a+b) c, S2 = sum a (d-c),
 *                      S3 = sum b (c+d), c = x'[cplus], d = x'[cminus]; plane + = S1 - S3, plane - = S1 + S2  (3/4 of mode 2's work)
 * on the tcgen05 tensor cores, Z generated on the fly into tensor memory (3-pass fp16 split, fp32 partial sums drained every
 * flush_stages (0 = default) stages of 64 K values).  w_img: se3_zgemm_pack of every segment in order.  Co % 128 == 0,
 * (Ci * F) % 4 == 0 (F = 1 for mode 1, else 2; mode 3: Ci % 4 == 0), <= 16 segments (HOST array).  out rows: edge stride out_edge_stride floats, plane c at comp_off{c}. */
int     se3_zgemm_tile_n(int Co, int mode);
int64_t se3_zgemm_image_bytes(int Co, int mode, int total_stages);
int se3_zgemm_pack(const float* Fp, int Kp, int col0, int Co, int CiF, int mode, int total_stages, int stage0, void* image, void* stream);
int se3_zgemm_fwd(const se3_zseg* segs, int n_seg, const void* w_img, const float* sx, int64_t E, int Co, int mode,
                  float* out, int64_t out_edge_stride, int comp_off0, int comp_off1, int flush_stages, void* stream);

/* Masked mean over the neighbour axis (utils.py:72-80): x [B, K, C] , mask [B, K] (NULL = plain mean) -> out [B, C]. */
int se3_pool_fwd(const float* x, const uint8_t* mask, int64_t B, int K, int64_t C, float* out, void* stream);

/* NormSE3 (S:97-152, non-gated): x, out [rows = b*n*C, M]; norm = max(||x[r,:]||, eps);
 * out[r,:] = f(norm * scale[r % C]) * x[r,:] / norm with f = exact-erf GELU (use_gelu != 0) or identity. */
int se3_norm_fwd(const float* x, const float* scale, int64_t rows, int C, int M, float eps, int use_gelu, float* out, void* stream);

/* Attention for one degree (S:476-517): for every node i and head h
 *   keys/values along j = [global (G) | null (0/1) | self (0/1) | K neighbours]  (prepend order of S:485,499,505)
 *   sim_j = scale * sum_{d,m} q[b,i,h,d,m] k_j[d,m];  masked neighbour -> -FLT_MAX (S:510-513); softmax over j; out = sum_j a_j v_j.
 * q, out: [b,n,H*Dh,M].  k, v: [b,n,K,Ckv,M] with Ckv = kv_heads*Dh, kv_heads in {H,1} (1 = OneHeadedKVAttentionSE3, S:643-651).
 * If k_idx != NULL, k is node level [b,n,Ckv,M] and neighbour j reads k[b, k_idx[b,i,j]] (linear_proj_keys, S:461-463).
 * self_k/self_v: [b,n,Ckv,M] or NULL; null_k/null_v: [Ckv,M] or NULL; global_k/global_v: [b,G,Ckv,M] or NULL.
 * nmask: [b,n,K] or NULL. */
int se3_attn_fwd(const float* q, const float* k, const float* v, const int64_t* k_idx,
                 const float* self_k, const float* self_v, const float* null_k, const float* null_v,
                 const float* global_k, const float* global_v, int G, const uint8_t* nmask,
                 int b, int n, int K, int H, int Dh, int M, int kv_heads, float scale, float* out, void* stream);

/* LinearSE3 (S:78-95) on the tensor cores: out[node, o, m] = sum_d x[node, d, m] W[d, o] (+ res[node, o, m]); x [nodes, D, M] and
 * out / res [nodes, Eo, M] in the reference layout (no transposed copies), 3-pass fp16 split with fp32 partial sums as in
 * se3_zgemm_fwd.  w_img = se3_zgemm_pack(Fp = W^T [Eo, D] viewed as [Eo * D/16, 16], Kp 16, col0 0, Co Eo, CiF D/16, mode 4,
 * total_stages D/64, stage0 0) (se3_zgemm_image_bytes(Eo, 4, D/64) bytes).  sx [nodes]: se3_pow2_scale_fwd of the row maxima
 * (se3_rowabsmax_fwd) with target exponent 14.  D % 64 == 0, Eo % 128 == 0.  res may be NULL. */
int se3_linear_tc_fwd(const float* x, const void* w_img, const float* res, const float* sx, int64_t nodes, int D, int Eo, int M,
                      float* out, void* stream);
/* sx[r] = power of two with rowmax[r] * sx[r] in [2^(target_exp-1), 2^target_exp) (1 for zero / non-finite rows). */
int se3_pow2_scale_fwd(const float* rowmax, int64_t rows, int target_exp, float* sx, void* stream);

/* As se3_attn_fwd for degrees >= 1 when the values (and, with k_aligned != 0, the keys) are still in the edge-aligned frame:
 * v (k) [b,n,K,M,Ckv] = the component-major out' of se3_zgemm_fwd, D [b*n*K, M, M] the frames of se3_frames_fwd,
 * k[e,d,:] = D(e) k'[e,:,d].  The rotation back to the global frame (se3_rotate_back / fold_basis of the unfused path) happens
 * inside the kernel, so the global-frame K / V tensors are never materialised.  With k_aligned == 0 the keys are in the
 * global frame as for se3_attn_fwd (node level with k_idx, linear_proj_keys).  Prefix keys/values (self, null, global) are
 * global-frame as before. */
int se3_attn_aligned_fwd(const float* q, const float* k, const float* v, const float* D, int k_aligned, const int64_t* k_idx,
                         const float* self_k, const float* self_v, const float* null_k, const float* null_v,
                         const float* global_k, const float* global_v, int G, const uint8_t* nmask,
                         int b, int n, int K, int H, int Dh, int M, int kv_heads, float scale, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SE3B200_H */
