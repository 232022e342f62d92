/*
 * hfl.h -- C ABI of libhfl_b200.so: the B200-native (sm_100a) kernels behind the
 * HOTFormerLoc embedding hot path  (raw lidar submaps -> batched octree ->
 * hierarchical octree transformer -> 256-d descriptor -> top-k retrieval).
 *
 * Conventions (SURVEY.md section 8b):
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`;
 *   - the caller owns every buffer, including workspaces (query the size with
 *     the matching *_workspace_bytes); kernels never allocate or free;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*),
 *     and re-entrant; the only process state is idempotent bookkeeping (a launch counter, the
 *     per-device "dynamic shared memory limit already raised" marks, environment toggles read once);
 *   - every call returns 0 on success or a negative hfl_status; nothing throws
 *     or aborts across the ABI.  hfl_last_error_string() is thread-local.
 *
 * Each entry point names the reference interface it replaces
 * (file:line under the reference tree; "ocnn" = third-party ocnn==2.2.2,
 * reference requirements.txt:7, restated in SURVEY.md Appendix A).
 */
#ifndef HFL_H_
#define HFL_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HFL_MAX_DEPTH 15
#define HFL_OK 0
#define HFL_ERR_INVALID (-1)   /* bad argument                                  */
#define HFL_ERR_CUDA (-2)      /* a CUDA runtime call / launch failed           */
#define HFL_ERR_WORKSPACE (-3) /* workspace too small                           */
#define HFL_ERR_UNSUPPORTED (-4)

const char* hfl_last_error_string(void);
int hfl_version(void);
/* number of kernels launched by this library in the calling process so far
 * (bench.py reports the delta over its timed region as "gpu_launches"). */
int64_t hfl_launch_count(void);

/* ------------------------------------------------------------------------
 * Batched octree (SURVEY.md section 8 rows a1-a4, a6)
 * ------------------------------------------------------------------------ */

/* Device-resident batched octree.  Node arrays are indexed by the rank of the
 * node among the NON-EMPTY nodes of its depth over the whole batch (the order
 * of ocnn.octree.merge_octrees).  `nkey[d]` holds the compact sort key
 *      (submap << 3d) | morton_d(x,y,z)          (x most significant per triple)
 * from which the reference's key ((submap << 48) | morton) is a bit move.
 * counts[d*(batch+2) + b] = nodes of submap b at depth d (batch_nnum_nempty),
 * counts[d*(batch+2) + batch]   = nnum_nempty[d],
 * counts[d*(batch+2) + batch+1] = nnum[d]. */
typedef struct hfl_octree {
  int32_t depth, full_depth, batch, _pad;
  int64_t n_points;
  int64_t cap[HFL_MAX_DEPTH + 1];       /* row capacity of nkey[d] / nidx[d]     */
  uint64_t* nkey[HFL_MAX_DEPTH + 1];    /* [cap[d]]                               */
  int32_t* children[HFL_MAX_DEPTH + 1]; /* [8*cap[d-1]] (d>full) | [batch*8^d]    */
  int32_t* nidx[HFL_MAX_DEPTH + 1];     /* [cap[d]] all-node index of each node   */
  float* leaf_points;                   /* [cap[depth]*3] mean point, octree units */
  int32_t* point_leaf;                  /* [n_points] or NULL: build_octree's idx */
  int32_t* counts;                      /* [(depth+1)*(batch+2)]                  */
} hfl_octree;

size_t hfl_octree_build_workspace_bytes(int64_t n_points, int32_t batch, int32_t depth);

/* Replaces, for a whole batch at once: ocnn Octree.build_octree (called at
 * eval/pnv_evaluate.py:173-175, datasets/dataset_utils.py:90-92) and
 * ocnn.octree.merge_octrees (eval/pnv_evaluate.py:123).
 * points: [n_points*3] fp32 in [-1,1], submaps packed back to back;
 * pt_offsets: [batch+1] int32 prefix offsets (device). */
int hfl_octree_build(const float* points, const int32_t* pt_offsets, const hfl_octree* out,
                     void* workspace, size_t workspace_bytes, void* stream);

/* An ocnn octree (SURVEY.md Appendix A) as the reference's collate_batch / to_device hand it to
 * the model (eval/pnv_evaluate.py:122-126, 173-176).  Counts are host values; arrays are device
 * arrays over ALL nodes of a depth:
 *   keys[d]     [nnum[d]] int64 (submap << 48) | morton_d
 *   children[d] [nnum[d]] int32 rank among the non-empty nodes of depth d, -1 if empty
 *   points      [nnum_nempty[depth]*3] fp32 leaf means in octree units (ocnn points[depth]). */
typedef struct hfl_ocnn_octree {
  int32_t depth, full_depth, batch, _pad;
  int64_t nnum[HFL_MAX_DEPTH + 1];
  int64_t nnum_nempty[HFL_MAX_DEPTH + 1];
  const int64_t* keys[HFL_MAX_DEPTH + 1];
  const int32_t* children[HFL_MAX_DEPTH + 1];
  const float* points;
} hfl_ocnn_octree;

/* Invariant bits of status[0] written by hfl_octree_import. */
#define HFL_IMPORT_BAD_CHILDREN 1 /* non-negative children[d] are not 0,1,..,nnum_nempty[d]-1 in order */
#define HFL_IMPORT_BAD_KEYS 2     /* keys[d] disagree with the node's position / its parent's key   */

/* Host only, touches no device memory: the count relations hfl_octree_import checks first,
 *   1 <= full_depth < depth <= 15, 1 <= batch < 32768, 0 <= nnum_nempty[d] <= nnum[d] < 2^31,
 *   nnum[d] == batch*8^d (d <= full_depth), nnum_nempty[d] == nnum[d] (d < full_depth),
 *   nnum[d] == 8*nnum_nempty[d-1] (d > full_depth).
 * With them, every structural index of the import (such as the parent i >> 3 of node i) is in range. */
int hfl_octree_import_check(const hfl_ocnn_octree* in);
size_t hfl_octree_import_workspace_bytes(const hfl_ocnn_octree* in);

/* Fills `out` (allocated for in->depth / full_depth / batch, cap[d] >= nnum_nempty[d] and
 * cap[d] == batch*8^d for d <= full_depth) from an ocnn octree, so that it holds what
 * hfl_octree_build writes for the same clouds: nkey, nidx, children, leaf_points and the counts
 * table; point_leaf is not touched (ocnn does not keep it).  The host-side count relations are
 * checked before any launch (HFL_ERR_INVALID).  The device-side invariants are checked by the
 * kernels: status [2] int32 receives status[0] = HFL_IMPORT_* bits of the violated invariants and
 * status[1] = a mask with bit d set for every depth d at which one failed.  Whatever the input,
 * every index the output holds is in range, so the neighbour / token kernels may run on it; its
 * values are meaningful only when status[0] == 0.  Lets HOTFormerLoc.forward
 * (models/hotformerloc.py:33) take the ocnn octree the reference's callers build. */
int hfl_octree_import(const hfl_ocnn_octree* in, const hfl_octree* out, int32_t* status,
                      void* workspace, size_t workspace_bytes, void* stream);

/* Replaces ocnn Octree.construct_neigh (misc/torch_utils.py:49-51).
 * Depth d <= full_depth: `grid` [batch*8^d*27] receives the full-grid table
 * (entries index ALL nodes), and na_out rows are gathered from it.
 * Depth d > full_depth: derived from na_parent = NA[d-1].
 *   na_out [cap[d]*27]: rows = non-empty nodes, entries = all-node indices
 *   ne_out [cap[d]*27] or NULL: same rows, entries = non-empty indices
 *          (== ocnn Octree.get_neigh(d,'333',stride=1,nempty=True),
 *           libs/dwconv/dwconv/nn.py:59, models/octree.py:95-110). */
int hfl_octree_neigh(const hfl_octree* o, int32_t d, const int32_t* na_parent, int32_t* grid,
                     int32_t* na_out, int32_t* ne_out, void* stream);

/* Reference-layout table for depth d: [nnum[d]*27] rows = ALL nodes (ocnn
 * Octree.neighs[d]); used for API parity and the batch_45.npz known answer. */
int hfl_octree_neigh_full(const hfl_octree* o, int32_t d, const int32_t* na_parent,
                          int32_t* full_out, void* stream);

/* ocnn Octree.keys[d] in the reference's int64 layout, [nnum[d]]. */
int hfl_octree_full_keys(const hfl_octree* o, int32_t d, int64_t* keys_out, void* stream);

/* Per-token (x,y,z,submap) int16x4 table padded to n_pad rows with (0,0,0,batch):
 * what models/octree.py:130-154, 272-283 derive through key2xyz / batch_id. */
int hfl_octree_tokens(const hfl_octree* o, int32_t d, int64_t n_pad, int16_t* xyzb_out,
                      void* stream);

/* ------------------------------------------------------------------------
 * Dense / gather kernels of the forward pass (SURVEY.md section 8 rows a5, a8-a15)
 * Activations: fp32 residual stream + bf16 shadow; weights bf16 [N, KD*Cin].
 * ------------------------------------------------------------------------ */

/* tcgen05 gather-GEMM with fused epilogue.
 *   v = sum_kk A[idx[m,kk], :] . W[:, kk*Cin:(kk+1)*Cin]^T (+bias) (+res[orow])  ; act: 1 = GELU
 *   y = LayerNorm(v) (ln_g/ln_b non-NULL, needs N <= 256) ; relu: ReLU after LN
 *   orow = out_rows ? out_rows[m] : m (negative: row skipped); y rows = orow if y_mapped else m
 * Replaces torch.nn.Linear (octformer_backbone.py:39-41, octformer_layers.py:48-59,
 * hotformerloc_backbone.py:72-74), ocnn.nn.OctreeConv (octformer_layers.py:89,
 * octformer_backbone.py:470: idx = get_neigh table, KD = 27 or 8) and the LayerNorm /
 * ReLU / residual adds around them. */
int hfl_gather_gemm(const void* A, const int32_t* idx, const void* W, int64_t M, int32_t N,
                    int32_t KD, int32_t Cin, const float* bias, const float* res, int32_t act,
                    float* out_v_f32, void* out_v_bf16, const float* ln_g, const float* ln_b,
                    int32_t relu, int32_t y_mapped, float* out_y_f32, void* out_y_bf16,
                    const int32_t* out_rows, void* stream);

/* Fused transformer MLP: out[orow] = res[orow] + fc2(GELU(fc1(A) + b1)) + b2, hidden never
 * leaves the SM.  W1: [4C, C] bf16, W2: [C, 4C] bf16 (nn.Linear layouts).  Replaces MLP.forward
 * (octformer_layers.py:53-59) + the residual add of the pre-LN blocks
 * (octformer_backbone.py:279-281, hotformerloc_backbone.py:215-216, 290-291). */
int hfl_mlp_fused(const void* A, const void* W1, const float* b1, const void* W2, const float* b2,
                  int64_t M, int32_t C, const float* res, float* out_f32, void* out_bf16,
                  const int32_t* out_rows, void* stream);

/* Attention output projection + residual + norm2 + MLP + residual in one kernel:
 *   s = res[orow] + O . Wp^T + bp ;  out[orow] = s + fc2(GELU(fc1(LayerNorm(s)) + b1)) + b2
 * O: [M, C] bf16 attention output (before proj), Wp: [C, C] bf16.  The projected tile, norm2 and the
 * hidden activation never leave the SM; the fp32 residual stream is read and written once.
 * Replaces `x = x + proj(attn)` + `x = x + mlp(norm2(x))` of the pre-LN blocks
 * (octformer_backbone.py:276-281, hotformerloc_backbone.py:212-216, 287-291). */
int hfl_proj_mlp_fused(const void* O, const void* Wp, const float* bp, const float* ln_g,
                       const float* ln_b, const void* W1, const float* b1, const void* W2,
                       const float* b2, int64_t M, int32_t C, const float* res, float* out_f32,
                       void* out_bf16, const int32_t* out_rows, void* stream);

/* Octree window attention core (octformer_backbone.py:52-93 + RPE octformer_layers.py:144-170):
 * softmax(q k^T * scale + [same-submap mask] + RPE) v per (window, head), head_dim 16.
 * Window w holds K tokens: plain rows w*K+s; dilated rows (w/dil)*K*dil + s*dil + w%dil;
 * hat: K+1 rows w*(K+1)+s with the relay token first.  rpe: [3*(2*bnd+1), H] or NULL. */
int hfl_window_attn(const void* qkv, void* out, const int16_t* xyzb, const float* rpe,
                    int64_t n_win, int32_t H, int32_t C, int32_t K, int32_t dil, int32_t hat,
                    int32_t bnd, float scale, void* stream);

/* Fused qkv projection + octree window attention (everything of OctreeAttention.forward before `proj`,
 * octformer_backbone.py:52-88): out = softmax(q k^T * scale + mask + RPE) v with q, k, v = y Wqkv^T + b
 * computed on chip (tcgen05: projection, q k^T and p v; the [rows, 3C] qkv tensor never exists).
 * y: [rows, C] bf16 LayerNorm'ed tokens in the window layout of hfl_window_attn.  Wg / bias_g: the
 * nn.Linear(C, 3C) weight [3C, C] bf16 / bias with rows regrouped per 4 heads as [q(64) | k(64) | v(64)]
 * (hotformerloc_b200.ops.regroup_qkv).  hfl_qkv_attn_supported() tells whether a configuration is
 * handled (window length K + hat in {16,17,32,33,48,49,64}, C in {128,256}); otherwise use
 * hfl_gather_gemm + hfl_window_attn. */
int hfl_qkv_attn_supported(int32_t H, int32_t C, int32_t K, int32_t dil, int32_t hat, int32_t bnd);
int hfl_qkv_attn(const void* y, const void* Wg, const float* bias_g, void* out, const int16_t* xyzb,
                 const float* rpe, int64_t n_win, int64_t rows, int32_t H, int32_t C, int32_t K, int32_t dil,
                 int32_t hat, int32_t bnd, float scale, const uint32_t* codes, void* stream);
/* Optional: the (query, key) pair codes of a level (clamped relative-position table offsets + the same-submap /
 * relay-token cases; models/layers/octformer_layers.py:144-163, models/octree.py:186-209).  They depend on the
 * token positions only, not on the block, so a caller running several blocks on one level makes them once
 * (hfl_qkv_attn_codes_bytes() bytes) and passes them to every hfl_qkv_attn of that level (with the same K, dil, hat,
 * bnd and rpe != NULL); with codes == NULL the kernel derives them per tile. */
int64_t hfl_qkv_attn_codes_bytes(int64_t n_win, int32_t K, int32_t hat);
int hfl_qkv_attn_codes(const int16_t* xyzb, int64_t n_win, int32_t K, int32_t dil, int32_t hat, int32_t bnd,
                       int32_t use_rpe, uint32_t* codes, void* stream);

/* Relay-token self-attention over ragged per-submap sequences
 * (hotformerloc_backbone.py:83-119 with the mask of models/octree.py:229-265). */
int hfl_varlen_attn(const void* qkv, void* out, const int32_t* cu_seqlens, const int32_t* ids,
                    int32_t B, int32_t max_len, int32_t H, int32_t C, float scale, void* stream);

/* InputFeature('P') + first OctreeConv 3^3 (3->32) + LayerNorm + ReLU
 * (hotformerloc.py:28-31, octformer_backbone.py:451-456). w: [81,32] fp32. */
int hfl_stem_conv(const float* leaf_pts, const int32_t* ne, int64_t n, int32_t depth,
                  const float* w, const float* g, const float* b, void* out_bf16, void* stream);

/* x += LayerNorm(dwconv27(x)) fused with the block's norm1 -> bf16 GEMM operand.
 * Replaces dwconv.core.dwconv_forward_backward (libs/dwconv/csrc/dwconv.cu:99-113,
 * pybind.cpp:10-14) + CPE norm (octformer_layers.py:138-142) + norm1.
 * K = 0: plain layout, else hat layout.  cpe_out != NULL: only LN(dwconv(x)) -> [n,C]. */
int hfl_cpe_ln(float* x, const void* xb, const int32_t* ne, const void* w_bf16, const float* g_cpe,
               const float* b_cpe, const float* g1, const float* b1, void* y1_bf16, float* cpe_out,
               int64_t n, int64_t rows, int32_t C, int32_t K, void* stream);

int hfl_ln_rows(const float* x, const int32_t* rows, int64_t m, int32_t C, const float* g,
                const float* b, void* y_bf16, void* stream);

/* Relay-token initialisation (hotformerloc_backbone.py:345-363), ADaPE window statistics
 * (models/octree.py:285-344) and ADaPE fc1+GELU (octformer_layers.py:203-210).
 * mode: 0 none | 3 pos | 6 var | 9 cov. */
int hfl_rt_init(float* x, const float* src, const int16_t* xyzb, int64_t n, int64_t n_win,
                int32_t K, int32_t C, int32_t depth, int32_t mode, const float* w1,
                const float* b1, void* h_bf16, float* stats_out, void* stream);

int hfl_hat_rows(int32_t* out, int64_t n, int32_t K, int32_t offset, void* stream);
int hfl_remap_hat(const int32_t* in, int32_t* out, int64_t n, int32_t K, void* stream);
int hfl_f32_to_bf16(const float* in, void* out, int64_t n, void* stream);

/* AdaptivePooling (salsa.py:25-55) given logits = x . query^T from hfl_gather_gemm. */
int hfl_attn_pool(const float* logits, const float* x, const void* x_bf16, const int32_t* tok_off,
                  float* stat, float* out, int32_t B, int32_t kq, int32_t ldl, int32_t K, int32_t C,
                  int32_t ktot, int32_t q_off, float scale, void* stream);

/* Mixer channel_proj + row_proj + flatten (salsa.py:105-111) + F.normalize (hotformerloc.py:55). */
int hfl_mixer_tail(const float* x, const float* wc, const float* bc, const float* wr,
                   const float* br, float* out, int32_t B, int32_t kin, int32_t kout, int32_t C,
                   int32_t od, int32_t normalize, void* stream);

/* PyramidOctGeM level pooling (pooling.py:92-96 + ocnn OctreeGlobalPool). */
int hfl_gem_pool(const float* x, const int32_t* tok_off, int32_t B, int32_t K, int32_t C, float pw,
                 float eps, float* out, int32_t ld_out, int32_t col_off, void* stream);

/* PyramidOctGeM descriptor head: Linear(no bias) + eval BatchNorm1d (+ L2 normalise), fp32
 * (pooling.py:78-84, 98-99). w: [out_dim, in_dim]. */
int hfl_gem_head(const float* pooled, int32_t B, int32_t in_dim, const float* w, const float* bn_g,
                 const float* bn_b, const float* bn_mean, const float* bn_var, float bn_eps,
                 int32_t out_dim, int32_t normalize, float* out, void* stream);

/* OPT-IN device-side form of the pre-octree transforms of the evaluation loop (eval/pnv_evaluate.py:158-171):
 * Normalize, bounding-box form (datasets/augmentation.py:212-235) -> |coord| <= 1 mask -> [radial mask ->
 * CylindricalCoordinates(use_octree=True), datasets/coordinate_utils.py:68-116] -> stable per-cloud compaction.
 * in: [n_in*3] raw fp32 points of B clouds back to back, off_in [B+1].  tmp: [n_in*3], cnt: [B] scratch.
 * out: [<= n_in*3] prepared points, off_out: [B+1] their offsets = the inputs of hfl_octree_build;
 * total_out (optional, e.g. mapped / pinned host memory): number of prepared points.
 * scale_factor > 0: coords / scale_factor, else coords * (2 norm_range / (max extent + 1e-6)).
 * Bit-identical to the host path except for sqrt / atan2, where torch's CPU kernels are not correctly rounded
 * (last-bit differences, see csrc/prep.cu and DESIGN.md section 6). */
int hfl_prepare_clouds(const float* in, const int32_t* off_in, int32_t B, int64_t n_in, int32_t norm,
                       int32_t zero_mean, float scale_factor, float norm_range, int32_t cyl, float* tmp,
                       int32_t* cnt, float* out, int32_t* off_out, int32_t* total_out, void* stream);

/* ------------------------------------------------------------------------
 * Octree depth-wise convolution with backward, fp32 (the reference's `dwconv.core`,
 * libs/dwconv/csrc/pybind.cpp:10-14; training-side, not called by the embedding path)
 * neigh: [rows, K] neighbour table, int64 (neigh_i64 != 0, the reference layout) or int32,
 * 1 <= K <= 27; an entry outside [0, n_in) (or [0, n_data)) is an empty tap.
 * ------------------------------------------------------------------------ */

/* out[i,c] = sum_k w[k,c] * data[neigh[i,k],c] over the non-empty taps; data [n_in, C], w [K, C]
 * ((K,1,C) in the reference), out [n_out, C].  Each element is accumulated from 0.f in ascending
 * k with fmaf, the order of the reference kernel.  With the inverse table (hfl_dwconv_inverse) in
 * place of neigh and the output gradient in place of data it is the input gradient.
 * Replaces dwconv_forward_backward (libs/dwconv/csrc/dwconv.cu:99-113). */
int hfl_dwconv(const float* data, const void* neigh, int32_t neigh_i64, const float* w, int64_t n_out,
               int64_t n_in, int32_t K, int32_t C, float* out, void* stream);

/* ineigh_out [n_data, K], same dtype as neigh: ineigh[neigh[i,k], k] = i, -1 where no row points.
 * A well-formed stride-1 octree table hits each (j,k) at most once; if several rows hit one (j,k)
 * the entry is the largest such i (deterministic, where the reference's scatter races).
 * Replaces inverse_neigh (libs/dwconv/csrc/dwconv.cu:74-85, :87). */
int hfl_dwconv_inverse(const void* neigh, int32_t neigh_i64, int64_t n_rows, int64_t n_data, int32_t K,
                       void* ineigh_out, void* stream);

/* dw[k,c] = sum_i grad[i,c] * data[neigh[i,k],c]; grad [n, C], neigh [n, K], dw [K, C].  Fixed-order
 * sums without float atomics over a row partition that depends on (n, K, C) only: bit-identical
 * across runs and GPUs.  ws: hfl_dwconv_wgrad_workspace_bytes(n, K, C) bytes, 16-byte aligned.
 * Replaces dwconv_weight_backward (libs/dwconv/csrc/dwconv.cu:45-72, :115). */
int64_t hfl_dwconv_wgrad_workspace_bytes(int64_t n, int32_t K, int32_t C);
int hfl_dwconv_wgrad(const float* grad, const float* data, const void* neigh, int32_t neigh_i64, int64_t n,
                     int64_t n_in, int32_t K, int32_t C, float* dw, void* ws, int64_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------
 * Octree window attention core with backward, fp32 (training side, not called by the embedding
 * path): OctreeAttention.forward from qkv to before proj, with the RPE bias, the submap mask and
 * the H-OSA relay token.  For window n, head h (head dim 16, C = 16 H, 1 <= H <= 16), queries i and
 * keys j of the L = K + hat window positions (1 <= L <= 128):
 *   s = (q_i . k_j) 0.25 + (ids[n,i] == ids[n,j] ? 0 : -1000)
 *       + sum_a rpe_table[clamp(x_ia - x_ja, -bnd, bnd) + bnd + a (2 bnd + 1), h]
 *   o[n,i,16h+e] = sum_j softmax_j(s) v[n,h,j,e]
 * With hat = 1 the relay token is position 0 and its row and column get no RPE term.
 *   qkv  [n_win, L, 3C] fp32, the output of Linear(C, 3C): column of (s, h, e) = s C + 16 h + e
 *   xyz  [n_win, L - hat, 3] int32 / int64 (xyz_i64) integer cell coordinates of the window tokens
 *        (after any dilation gather); may be NULL when rpe_table is NULL
 *   ids  [n_win, L] int32 / int64 (ids_i64); tokens attend with bias 0 iff their ids are equal
 *   rpe_table [3 (2 bnd + 1), H] fp32 or NULL (no RPE), 0 <= bnd <= 2^20
 *   o    [n_win, L, C] fp32, lse [n_win, H, L] fp32 (per-row log-sum-exp, kept for the backward)
 * qkv, o, dout and dqkv must be 16-byte aligned.  No [n_win, H, L, L] tensor is written.
 * ------------------------------------------------------------------------ */

/* Replaces OctreeAttention.forward's core (octformer_backbone.py:52-93), the RPE gather
 * (octformer_layers.py:156-170) and HOTFormerBlock's relay-token attention (hotformerloc_backbone.py:197-236). */
int hfl_window_attn_train_fwd(const float* qkv, const void* xyz, int32_t xyz_i64, const void* ids, int32_t ids_i64,
                              const float* rpe_table, int64_t n_win, int32_t L, int32_t H, int32_t hat, int32_t bnd,
                              float* o, float* lse, void* stream);

/* Backward of hfl_window_attn_train_fwd (octformer_backbone.py:52-93, octformer_layers.py:156-170,
 * hotformerloc_backbone.py:197-236 under autograd): given dout [n_win, L, C] and the forward's o and
 * lse, writes dqkv [n_win, L, 3C] and, with a table, drpe_table [3 (2 bnd + 1), H] (three bins per
 * token pair, nothing from the relay token's row or column).  Every dqkv element is a fixed-order
 * fp32 sum; the table gradient is summed in exact int64 fixed point (range argument in
 * csrc/window_attn_train.cu).  Both are bit-identical across runs, without float atomics.
 * ws: hfl_window_attn_train_bwd_workspace_bytes(H, bnd, rpe_table != NULL) bytes, 256-byte aligned
 * (0 bytes and NULL without a table). */
int64_t hfl_window_attn_train_bwd_workspace_bytes(int32_t H, int32_t bnd, int32_t has_rpe);
int hfl_window_attn_train_bwd(const float* qkv, const void* xyz, int32_t xyz_i64, const void* ids, int32_t ids_i64,
                              const float* rpe_table, const float* o, const float* lse, const float* dout,
                              int64_t n_win, int32_t L, int32_t H, int32_t hat, int32_t bnd, float* dqkv,
                              float* drpe_table, void* ws, int64_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------
 * Attention pooling over ragged per-submap token segments with backward, fp32 (training side, not
 * called by the embedding path): the AdaptivePooling of PyramidAttnPoolWrapper without the padded
 * (B, Nmax, C) features and the (B, N, N) mask.  Segment b = tokens [offsets[b], offsets[b+1]) of
 * x [n, C]; queries Q [k, C]; s = C^-0.5:
 *   S[b,q,t] = s Q[q].x[t]     out[b,q] = sum_t softmax_t(S[b,q,.]) x[t]     lse[b,q] = log sum_t exp(S[b,q,t])
 * An empty segment gives out = 0 and lse = -inf, and contributes no gradient.
 *   offsets [B+1] int64 (device); each entry is clamped into [0, n] and a decreasing pair is an empty
 *           segment, so no offsets value makes a kernel access memory out of range.  The results are
 *           those of the formula when the offsets are non-decreasing with offsets[0] = 0 and
 *           offsets[B] = n (every token in exactly one segment).
 *   1 <= k <= 256, C a multiple of 32 in [32, 512], n >= 0, 1 <= B <= 2^24;
 *   x, Q, dout 16-byte aligned; out, dout [B, k, C]; lse [B, k]; dx [n, C]; dQ [k, C].
 * Tokens are cut into segment-aligned chunks of 1024; the partition depends on (offsets, k, C) only
 * and every output element is a fixed-order fp32 sum (no float atomics, no TF32): out, lse, dx and dQ
 * are bit-identical across runs.  Workspaces: the *_workspace_bytes of (n, B, k, C), 256-byte
 * aligned, (ceil(n / 1024) + B) k (C + 2) 4 bytes forward and (ceil(n / 1024) + B) k C 4 bytes
 * backward, plus O(B k).
 * ------------------------------------------------------------------------ */
int64_t hfl_attn_pool_train_fwd_workspace_bytes(int64_t n, int32_t B, int32_t k, int32_t C);
int64_t hfl_attn_pool_train_bwd_workspace_bytes(int64_t n, int32_t B, int32_t k, int32_t C);

/* Replaces the split / pad of the local features to (B, Nmax, C), the (B, N, N) int64 mask and the
 * single-head attention of the learned queries (models/layers/pooling.py:183-233, salsa.py:25-55). */
int hfl_attn_pool_train_fwd(const float* x, const int64_t* offsets, const float* Q, int64_t n, int32_t B, int32_t k,
                            int32_t C, float* out, float* lse, void* ws, int64_t ws_bytes, void* stream);

/* Backward of hfl_attn_pool_train_fwd (pooling.py:183-233, salsa.py:25-55 under autograd): given dout
 * and the forward's out and lse, writes dx = sum_q p dout[b,q] + s sum_q dS Q[q] and
 * dQ = s sum_t dS x[t], with dS = p (dout[b,q].x[t] - dout[b,q].out[b,q]) and p recomputed from x, Q
 * and lse. */
int hfl_attn_pool_train_bwd(const float* x, const int64_t* offsets, const float* Q, const float* out,
                            const float* lse, const float* dout, int64_t n, int32_t B, int32_t k, int32_t C,
                            float* dx, float* dQ, void* ws, int64_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------
 * Relay-token self-attention core with backward, fp32 (training side, not called by the embedding
 * path): RTAttention.forward from qkv to before proj over the ragged per-submap RT sequences, without
 * concat_and_pad_rt's (B, Nmax, C) tensors and the (B, Nmax, Nmax) mask.  Sequence b = packed rows
 * [cu[b], cu[b+1]) of T; for head h (head dim 16, C = 16 H, 1 <= H <= 16) and rows i, j of one sequence:
 *   s_ij = 0.25 q_i.k_j + (ids[i] == ids[j] ? 0 : -1000)
 *   o[i, 16h+e] = sum_j softmax_j(s_i.) v_j[e]          lse[i, h] = log sum_j exp(s_ij)
 * The reference's padding slots carry -1000 against every real RT, so their weight is exactly 0 in
 * fp32 and the ragged form equals the padded one at every real row.
 *   qkv [T, 3C] fp32, the output of Linear(C, 3C): column of (s, h, e) = s C + 16 h + e
 *   cu  [B+1] int32 (device); each entry is clamped into [0, T] and never below the previous entry's
 *       clamped value, so a decreasing pair is an empty sequence, an entry above T cuts its sequence at
 *       T, sequences never overlap, and no cu value makes a kernel access memory out of range.  Rows in
 *       no sequence are not written.  A sequence may have any length from 0 to T.
 *   ids [T] int32 / int64 (ids_i64); rows attend with bias 0 iff their ids are equal (any values)
 *   o [T, C], lse [T, H], dout [T, C], dqkv [T, 3C] fp32; qkv, o, dout and dqkv 16-byte aligned
 *   1 <= B <= 2^24, T >= 0 with 3 C T < 2^31
 * Every output element is a fixed-order fp32 sum (no float atomics, no TF32): o, lse and dqkv are
 * bit-identical across runs.  ws: hfl_rt_attn_train_workspace_bytes(T, B, H) bytes, 256-byte aligned
 * (2 (B + 1) + T H 4-byte words, rounded up), for the forward and the backward alike.
 * ------------------------------------------------------------------------ */
int64_t hfl_rt_attn_train_workspace_bytes(int64_t T, int32_t B, int32_t H);

/* Replaces RTAttention.forward's core (hotformerloc_backbone.py:83-119) with the mask of
 * models/octree.py:229-265, and the padding of concat_and_pad_rt (relay_token_utils.py:12-40). */
int hfl_rt_attn_train_fwd(const float* qkv, const int32_t* cu, const void* ids, int32_t ids_i64, int32_t B,
                          int64_t T, int32_t H, float* o, float* lse, void* ws, int64_t ws_bytes, void* stream);

/* Backward of hfl_rt_attn_train_fwd (hotformerloc_backbone.py:83-119 under autograd): given dout and the
 * forward's o and lse, writes dqkv: with D_i = dO_i.o_i and p = exp(s - lse) recomputed from qkv,
 * dq_i = 0.25 sum_j p_ij (dO_i.v_j - D_i) k_j by query rows, then dk_j = 0.25 sum_i dS_ij q_i and
 * dv_j = sum_i p_ij dO_i by key rows over the queries of the key's own sequence. */
int hfl_rt_attn_train_bwd(const float* qkv, const int32_t* cu, const void* ids, int32_t ids_i64, const float* o,
                          const float* lse, const float* dout, int32_t B, int64_t T, int32_t H, float* dqkv, void* ws,
                          int64_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------
 * Octree convolution with backward, fp32 without TF32 (training side, not called by the embedding path):
 * ocnn.nn.OctreeConv for kernel 333 / stride 1 and kernel 222 / stride 2, nempty.
 *   neigh [n_out, K] int32 / int64 (neigh_i64), K in {8, 27}; an entry outside [0, n_in) is an empty tap
 *   data [n_in, Cin], w [K, Cin, Cout] (ocnn's `weights`), out [n_out, Cout]; 1 <= Cin, Cout <= 256
 * Work follows the occupied (row, tap) pairs: per tile of 128 output rows and tap the rows holding the
 * tap are compacted on the device before the tap's product runs.  Every output element is a fixed-order
 * fp32 sum (no float atomics): results are bit-identical across runs, GPUs and table dtypes.  The
 * rounding chains are documented in csrc/octree_conv_train.cu.
 * ------------------------------------------------------------------------ */

/* out[i,:] = sum_k sum_c data[neigh[i,k],c] w[k,c,:] over the occupied taps.  With the inverse table
 * (hfl_dwconv_inverse over neigh with n_data = n_in: stride 1 inv[j,k] = i where neigh[i,k] = j; stride 2
 * each input row's parent at its child position), the per-tap transposed weights [K, Cout, Cin] and the
 * output gradient in place of data it is the input gradient.
 * Replaces ocnn.nn.OctreeConv (octformer_layers.py:80-98 / :89, octformer_backbone.py:451-477 / :470). */
int hfl_octree_conv_train_fwd(const float* data, const void* neigh, int32_t neigh_i64, const float* w, int64_t n_out,
                              int64_t n_in, int32_t K, int32_t Cin, int32_t Cout, float* out, void* stream);

/* dw[k] = sum_i data[neigh[i,k]]^T (x) dout[i] over the occupied pairs; dout [n, Cout], dw [K, Cin, Cout].
 * Rows are cut into chunks that depend on (n, K, Cin, Cout) only; per-chunk partials go to ws and are
 * folded in chunk order.  ws: hfl_octree_conv_train_wgrad_workspace_bytes(n, K, Cin, Cout) bytes, 16-byte
 * aligned (at most 128 MiB).  n = 0 writes zeros.
 * Replaces the weight gradient of ocnn.nn.OctreeConv (octformer_layers.py:80-98 / :89,
 * octformer_backbone.py:451-477 / :470) under autograd. */
int64_t hfl_octree_conv_train_wgrad_workspace_bytes(int64_t n, int32_t K, int32_t Cin, int32_t Cout);
int hfl_octree_conv_train_wgrad(const float* data, const void* neigh, int32_t neigh_i64, const float* dout, int64_t n,
                                int64_t n_in, int32_t K, int32_t Cin, int32_t Cout, float* dw, void* ws,
                                int64_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------
 * Relay-token initialisation with backward, fp32 (training side, not called by the embedding path):
 * RelayTokenInitialiser.forward (hotformerloc_backbone.py:345-363) and the ADaPE window statistics of
 * OctreeT.compute_window_stats (models/octree.py:285-344).  Window w = rows [w K, (w + 1) K) of
 *   xyzb [n_win K, 4] int16 (x, y, z, submap), Octree.tokens(depth, n_win K): padding rows are (0, 0, 0, B)
 *   src  [n, C] fp32, the level's tokens; rows n <= t < n_win K are padding and count as zeros
 * A row is valid when its submap equals the window's first row's; cnt = number of valid rows (>= 1).
 *   rt_out [n_win, C]:  rt[w] = (sum of src over the valid rows) / cnt  (0 for an all-padding window)
 *   stats_out [n_win, mode] with mode 3 'pos' | 6 'var' | 9 'cov' (0: none, stats_out unused): the mean of
 *     the node centres xyz 2^(1-depth) - 1 (set to 0 at padding rows after the rescale) over max(cnt, 1),
 *     then the variances ('var') or upper-triangle covariances xx xy xz yy yz zz ('cov') with Bessel's
 *     correction max(cnt - 1, 1), zeroed unless cnt >= 2.  The statistics carry no gradient.
 * C a multiple of 32 in [32, 512]; 1 <= K <= 4096; 0 <= n <= n_win K; xyzb 8-byte aligned.
 * Fixed-order sums, no atomics: bit-identical across runs.
 * ------------------------------------------------------------------------ */
int hfl_rt_init_train_fwd(const float* src, const int16_t* xyzb, int64_t n, int64_t n_win, int32_t K, int32_t C,
                          int32_t depth, int32_t mode, float* rt_out, float* stats_out, void* stream);

/* Backward of hfl_rt_init_train_fwd: grad_src [n, C], grad_src[t] = grad_rt[w(t)] / cnt[w(t)] at the valid
 * rows and 0 at the others.  Each row lies in exactly one window, so it is a gather. */
int hfl_rt_init_train_bwd(const float* grad_rt, const int16_t* xyzb, int64_t n, int64_t n_win, int32_t K, int32_t C,
                          float* grad_src, void* stream);

/* Exact L2 top-k (eval/pnv_evaluate.py:200-225, 245) on one database shard, and the
 * merge of all-gathered partial lists. */
int hfl_knn_topk(const float* q, int32_t nq, const float* db, int32_t ndb, int32_t dim, int32_t k,
                 int32_t idx_offset, float* out_d, int32_t* out_i, void* stream);
/* Same with a caller-owned workspace of hfl_knn_workspace_bytes(): the database shard is split over the grid
 * (sorted partial lists per split, folded by the merge kernel) so that small query sets fill the GPU too. */
int64_t hfl_knn_workspace_bytes(int32_t nq, int32_t ndb, int32_t k);
int hfl_knn_topk_ws(const float* q, int32_t nq, const float* db, int32_t ndb, int32_t dim, int32_t k,
                    int32_t idx_offset, float* out_d, int32_t* out_i, void* ws, int64_t ws_bytes, void* stream);
int hfl_topk_merge(const float* in_d, const int32_t* in_i, int32_t parts, int32_t nq, int32_t k,
                   float* out_d, int32_t* out_i, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HFL_H_ */
