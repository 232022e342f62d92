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
