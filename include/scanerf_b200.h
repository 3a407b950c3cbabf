/*
 * scanerf_b200.h -- C ABI of libscanerf_b200.so, the drop-in boundary of the
 * B200-native (sm_100a) ScaNeRF hot path.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host;
 *   - row-major, dense (contiguous) arrays; shapes are given in the comments;
 *   - outputs are written in place into caller-allocated memory, elements the
 *     reference leaves untouched (sentinel fills) are left untouched here too;
 *   - `stream` is a cudaStream_t (NULL = legacy default stream, which is what the
 *     reference launches on);
 *   - return value 0 = launched; otherwise a cudaError_t, and snrf_last_error()
 *     returns a thread-local description.  Asynchronous faults surface at the next
 *     synchronisation, as with the reference's AT_CUDA_CHECK(cudaGetLastError()).
 * Each entry point cites the reference interface (file:line under the reference
 * checkout) it replaces.
 */
#ifndef SCANERF_B200_H
#define SCANERF_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- library ---------------------------------------------------------------- */
const char* snrf_last_error(void);
int snrf_version(void);
int snrf_device_sm_count(void);
/* L2 fetch granularity of the current device (cudaLimitMaxL2FetchGranularity; 32 / 64 / 128 bytes, a hint): bytes > 0 sets it,
 * bytes <= 0 only queries; returns the value in effect or a negative CUDA error code.  No reference counterpart: the
 * reference never touches the limit (hash-table gathers fetch one 32-byte sector per corner) */
int snrf_l2_fetch_granularity(int bytes);

/* ---- hash-grid encode ------------------------------------------------------- */
/* hashgrid/include/hashgrid.h:19-25 (embedding_forward_cuda, corner/size != NULL) and
 * :38-42 (embedding_bg_forward_cuda, corner = size = NULL).
 * points[B,3] f32, table[L,T,2] f32 (T power of two), res[L,3] i32, corner[3], size[3]
 * -> out[B,L,2] f32 (out_bf16=0) or out[B,2L] bf16 (out_bf16=1, tensor-core MLP input).
 * idx_out (optional) [B,L,8] u32: the hashed table indices of the 8 cell corners. */
int snrf_hash_fwd(const float* points, const float* table, const int* res, const float* corner,
                  const float* size, void* out, unsigned* idx_out, int B, int L, int T, int out_bf16,
                  void* stream);
/* hashgrid/include/hashgrid.h:27-35 / :45-51 (embedding_backward_cuda, embedding_bg_backward_cuda).
 * grad_in[B,L,2]; ACCUMULATES into grad_points[B,3] (may be NULL: skip d/dx) and
 * grad_table[L,T,2].  aggregate_levels: levels [0,n) use the warp-aggregated scatter
 * (-1 = default L/2). */
int snrf_hash_bwd(const float* points, const float* grad_in, const float* table, const int* res,
                  const float* corner, const float* size, float* grad_points, float* grad_table,
                  int B, int L, int T, int aggregate_levels, void* stream);
/* tuning hook: force the number of levels walked per CTA row (0 = automatic) */
void snrf_hash_set_levels_per_block(int lpb);

/* ---- fused training-path field encode -------------------------------------------- */
/* sample position -> space contraction -> hash encode in one kernel, replacing hashgrid/__init__.py:522
 * (samples = o + z d), :394-411 (contract_fore / contract_bg) and hashgrid/PyHashGridBG.py:9-30 with
 * hashgrid/src/hashgrid_bg_kernel.cu:106-275, plus their autograd.
 * mode 0: points[N,3] already contracted; mode 1 (fore) / 2 (background): sample n = rays_o[n/S] + z_vals[n] rays_d[n/S],
 * contracted w.r.t. the box (box_min, box_size: device float[3]); mode 3: rays [0, split) fore, rays [split, R) background
 * (both render chains of a step in one launch: the table streams through L2 once).
 * -> out_lm [L][N] float2 (level-major), jac_lm [L][3][N] float2 = d out / d contracted point (NULL: not needed). */
int snrf_field_encode_fwd(const float* rays_o, const float* rays_d, const float* z_vals, const float* points,
                          const float* box_min, const float* box_size, int mode, const float* table, const int* res,
                          float* out_lm, float* jac_lm, const unsigned char* ray_valid, int split, int N, int S, int L, int T,
                          void* stream);
/* grad_lm [L][N] float2, jac_lm from the forward (NULL: table gradient only).  ACCUMULATES grad_table [L,T,2] and
 * grad_rays_o / grad_rays_d [R,3] (modes 1, 2; either may be NULL) or grad_points [N,3] (mode 0). */
int snrf_field_encode_bwd(const float* rays_o, const float* rays_d, const float* z_vals, const float* points,
                          const float* box_min, const float* box_size, int mode, const int* res, const float* grad_lm,
                          const float* jac_lm, float* grad_rays_o, float* grad_rays_d, float* grad_points, float* grad_table,
                          const unsigned char* ray_valid, int split, int N, int S, int L, int T, void* stream);
/* The same backward FUSED with the sparse Adam update of the table (cuda/adam_kernel.cu:23-94 semantics: elements whose
 * gradient is exactly zero are skipped): the gradient of one L2-resident slice of the table at a time is scattered into
 * grad_scratch and consumed by the update on the spot, so no [L,T,2] gradient ever exists in HBM.  Equivalent to
 * snrf_field_encode_bwd into a zeroed gradient table followed by snrf_adam_step(..., step, zero_grad = 1).
 * table / exp_avg / exp_avg_sq [L,T,2] UPDATED in place; grad_rays_o / grad_rays_d / grad_points ACCUMULATED.
 * grad_scratch: scratch_entries float2, ALL ZERO on entry, left all zero: 2^23 (64 MiB, one L2-resident slice) is enough;
 * with T + 2^23 entries the levels [0, small_levels) -- those with few grid vertices, (rx+1)(ry+1)(rz+1) <= 2^22, whose
 * touched set is small whatever T is -- are reduced in one pass over the whole level instead of index range by index range;
 * cpts_scratch: 3 * N floats, overwritten (contracted sample positions, SoA). */
int snrf_field_encode_bwd_adam(const float* rays_o, const float* rays_d, const float* z_vals, const float* points,
                               const float* box_min, const float* box_size, int mode, const int* res, const float* grad_lm,
                               const float* jac_lm, float* grad_rays_o, float* grad_rays_d, float* grad_points,
                               float* table, float* exp_avg, float* exp_avg_sq, float lr, float beta1, float beta2, float eps,
                               int step, float* grad_scratch, long long scratch_entries, int small_levels, float* cpts_scratch,
                               const unsigned char* ray_valid, int split, int N, int S, int L, int T, void* stream);
/* Surface normals of the density field at every sample, forward only: replaces the out_normal branch of
 * HashGrid.render_batch_rays (hashgrid/__init__.py:547-556: torch.autograd.grad of sigma w.r.t. the samples, create_graph).
 * feats_lm [16][N] float2 and jac_lm [16][3][N] float2 from snrf_field_encode_fwd of the same rays (mode 1 = fore, 2 =
 * background; box_min, box_size, rays_o, rays_d [R,3], z_vals [R,S] as there); mask32 [32] (NULL = ones); params as
 * snrf_decoder_fwd (only Spatial_MLP.mlp.0, .mlp.2 and sigma_layer are read).  g = d sigma / d x at x = o + z d:
 * -> normal [N,3] = -g / (|g| + 1e-8), grad_x [N,3] = g (may be NULL).  fp32; softplus' as torch's (threshold 20); the
 * background contraction's max is differentiated at its arg-max axis, as torch.max is.  ray_valid (optional, bytes [R]):
 * rows of rays with a 0 flag are left untouched.  Grid-stride launch of min(ceil(N / 256), 2 x SMs) CTAs of 256 threads. */
int snrf_field_normal(const float* feats_lm, const float* jac_lm, const float* mask32, const float* const* params, int mode,
                      const float* box_min, const float* box_size, const float* rays_o, const float* rays_d,
                      const float* z_vals, const unsigned char* ray_valid, float* normal, float* grad_x, int N, int S,
                      void* stream);
/* measurement hook: when on, snrf_field_encode_bwd_adam times its three kernel classes with CUDA events (and SYNCHRONISES
 * the stream); snrf_field_last_profile -> out4 = milliseconds {geometry + ray gradient, scatter slices, Adam slices, both} */
void snrf_field_set_profile(int on);
void snrf_field_last_profile(float* out4);   /* [3] = the scatter + Adam phase as a whole (the only split available with the overlap on) */
/* tuning hook: 1 = the scatter of slice k+1 runs concurrently with the Adam of slice k (private side stream, the scratch
 * used as two halves); 0 (default; measured faster per byte of scratch) = strictly serial on the caller's stream */
void snrf_field_set_overlap(int on);
/* tuning hooks: run the single-pass coarse levels on a private side stream next to the other levels (default 1);
 * log2 of the entries of one L2-resident slice (default 23) */
void snrf_field_set_coarse_concurrent(int on);
/* tuning hook: L2 evict_last cache policy on the scratch accesses of the scatter + update fusion (default 1) */
void snrf_field_set_l2_hints(int on);
void snrf_field_set_slice_log2(int bits);
/* kernels launched by the last snrf_field_encode_bwd_adam call (1 + 2 per table slice) */
int snrf_field_last_launch_count(void);
/* tuning hook: cap on whole levels per scatter / update pair of snrf_field_encode_bwd_adam (0 = as many as fit the scratch) */
void snrf_field_set_levels_per_group(int n);
/* tuning hook: log2 of the number of table index ranges the scatter walks per level (-1 = automatic) */
void snrf_field_set_passes_log2(int bits);
/* tuning hook: levels [0, n) merge equal-cell lanes of a warp before reducing (-1 = automatic, L / 2) */
void snrf_field_set_aggregate_levels(int n);
/* tuning hook: kernels behind snrf_field_encode_bwd: 1 (default) = geometry / ray-gradient kernel + slim scatter per level and index
 * range (the pair of snrf_field_encode_bwd_adam, writing into grad_table), 0 = the round-1 single kernel */
void snrf_field_set_bwd_impl(int v);
/* tuning hook (experiment): the forward's CTA rows walk level pairs (y, L-1-y) instead of single levels (default 0) */
void snrf_field_set_fwd_pairing(int on);
/* tuning hook: L2 eviction policy of the forward's table gathers when a CTA row walks one level (large tables).
 * mode 0 = default policy; 1 = evict_last on every gather; 2 = the first pin_mib MiB of each level slice evict_last, the
 * rest evict_first; 3 = evict_last on the fraction pin_mib / 128 of the gathers, evict_first on the rest */
void snrf_field_set_fwd_l2_policy(int mode, int pin_mib);
/* tuning hook: x-pair gathers of the forward on levels >= first_level.  mode 0 = eight 8-byte loads per sample and level; 1 = one
 * 16-byte load for an x-pair in an aligned 16-byte slot; 2 = one 32-byte sector load per x-pair, the second corner fetched by
 * itself when it lies in another sector.  Results are bit-identical in every mode */
void snrf_field_set_fwd_pair_loads(int mode, int first_level);
/* measurement hook: unused dynamic shared memory (<= 48 KB) per CTA of the scatter / Adam slices = a cap on their resident CTAs */
void snrf_field_set_occupancy_smem(int bytes);
/* tuning hook: 1 (default) = the scatter / Adam slices of snrf_field_encode_bwd_adam are launched with the programmatic-stream-
 * serialization attribute (a slice's CTAs are scheduled while the previous slice drains and wait in `griddepcontrol.wait`) */
void snrf_field_set_pdl(int on);
/* tuning hook (experiment, default 0 = off): MiB of hardware L2 set-aside for which the gradient scratch of
 * snrf_field_encode_bwd_adam is a persisting access-policy window of its slice launches */
void snrf_field_set_persist_mib(int mib);
/* measurement hook: one forward launch per level, so that ncu reports L2 hit rate / DRAM bytes per level (default 0) */
void snrf_field_set_fwd_split_levels(int on);
/* tuning hook: samples per thread of the run-merging scatter kernel (2, 4 or 8; 0 selects the cross-lane kernel) */
void snrf_field_set_run_length(int r);

/* ---- bundle-adjustment pose chain -------------------------------------------------- */
/* camera_utils.py:86-89 (CAM.get_rts) + camera.py:84-95, 118-141 (Lie.se3_to_SE3, Taylor series) + camera.py:37-60
 * (Pose.compose_pair / invert): se3_refine [N,6], base_w2c [N,12] -> c2w [N,12] = invert(se3_to_SE3(se3) then base). */
int snrf_pose_fwd(const float* se3_refine, const float* base_w2c, float* c2w, int n, void* stream);
/* analytic backward of the above: grad_c2w [N,12] -> grad_se3 [N,6] (written) */
int snrf_pose_bwd(const float* se3_refine, const float* base_w2c, const float* grad_c2w, float* grad_se3, int n, void* stream);

/* ---- rays, boxes, samplers -------------------------------------------------- */
/* cuda/include/compute_ray.h (compute_ray_forward): Ks[N,9], C2Ws[N,12], locs[B,3] i32
 * = (view, px, py) -> rays_o, rays_d [B,3]. */
int snrf_compute_ray_fwd(float* rays_o, float* rays_d, const float* Ks, const float* C2Ws,
                         const int* locs, int B, void* stream);
/* cuda/include/compute_ray.h (compute_ray_backward): accumulates grad_C2Ws[N,12].
 * ref_index_bug=1 reproduces cuda/compute_ray_kernel.cu:71-72 (gradients read at view_idx). */
int snrf_compute_ray_bwd(const float* grad_o, const float* grad_d, const float* Ks, float* grad_C2Ws,
                         const int* locs, int B, int ref_index_bug, void* stream);
/* cuda/include/helper.h (ray_aabb_intersection K=1, ray_aabb_intersection_v2):
 * centers[K,3], sizes[K,3] (full extents) -> bounds[B,K,2] = (near,far) or (-1,-1). */
int snrf_ray_aabb(const float* rays_o, const float* rays_d, const float* centers, const float* sizes,
                  float* bounds, int B, int K, void* stream);
/* HashGrid.inverse_z_sampling + invalid_sampling_underground (hashgrid/__init__.py:287-293, 305-337; torch ops in
 * the reference): background samples z = 1 / (1 / (far + 1e-6) (1 - t) + t / 1e6) from the exit of the box
 * (center[3], size[3] full extents; far = 0.1 when the ray misses it), t_lin [S] = linspace(0, 1, S);
 * dists = forward differences (last 1e-6); valid [B] bytes (optional) = the exit is not on the floor face
 * (invalid_underground != 0) or all ones.  Bit-identical to the torch expression. */
int snrf_bg_inverse_z(const float* rays_o, const float* rays_d, const float* center, const float* size, const float* t_lin,
                      float* z_vals, float* dists, unsigned char* valid, int B, int S, int invalid_underground, void* stream);
/* cuda/include/helper.h (sample_points_grid): occupied[2^lx,2^ly,2^lz] bytes, log2dim[3] i32
 * (device) -> z_vals, dists [B,S]; counts[B] i32 optional (occupied segments per ray). */
int snrf_sample_grid(const float* rays_o, const float* rays_d, float* z_vals, float* dists,
                     const float* corner, const float* size, const unsigned char* occupied,
                     const int* log2dim, int* counts, int B, int S, void* stream);
/* cuda/include/sample.h (background_sampling_cuda) */
int snrf_bg_sampling(const float* starts, const float* bg_depth, float* z_vals, int B, int S,
                     float sample_range, void* stream);
/* cuda/include/sample.h (sample_insideout_block); *miss_flag set to 1 if any ray misses the box */
int snrf_sample_insideout(const float* rays_o, const float* rays_d, int S, int Sbg, const float* center,
                          const float* size, float far, float* z_vals, float* z_vals_bg, int* miss_flag,
                          int B, void* stream);

/* ---- front-to-back compositing ------------------------------------------------ */
/* hashgrid/__init__.py:344-366,564-596 (HashGrid.cal_integrate_weight / accumulate / tail of
 * render_batch_rays), which the reference runs as a chain of torch ops.
 * Per-sample heads are addressed base + n*stride (strides in floats): sigma[R*S], tint,
 * diffuse, specular [R*S,3]; z_vals, dists [R,S]; rays_d [R,3] (|d| scales the step).
 * -> weights[R,S], trans[R,S] (transmittance before each sample; may be NULL in fwd),
 *    out[R,16] = depth, tint3, diffuse3, specular3 (= sum w tint*spec), l2_3 (= sum w spec^2),
 *    T_left, 2 pad.  infinity != 0: the last step of rays r >= inf_start is 1e10.  ray_valid (optional, bytes [R]): rays with a 0 flag get
 *    zero weights / outputs and T_left = 1 (the defaults HashGrid scatters back for rays it did not render). */
int snrf_composite_fwd(const float* sigma, const float* tint, const float* diffuse, const float* specular,
                       int s_sigma, int s_tint, int s_diffuse, int s_specular,
                       const float* z_vals, const float* dists, const float* rays_d, const unsigned char* ray_valid,
                       int R, int S, int infinity, int inf_start, float* weights, float* trans, float* out, void* stream);
/* backward of the above: g_out[R,16] (same row layout; l2 columns act on specular only, the
 * weights inside l2 are detached as in the reference), g_weights[R,S] optional.  WRITES the
 * per-sample head gradients (strides gs_*) and grad_rays_d[R,3] (optional). */
int snrf_composite_bwd(const float* sigma, const float* tint, const float* diffuse, const float* specular,
                       int s_sigma, int s_tint, int s_diffuse, int s_specular,
                       const float* z_vals, const float* dists, const float* rays_d, const float* trans,
                       const float* g_out, const float* g_weights, const unsigned char* ray_valid, int R, int S, int infinity,
                       int inf_start, float* g_sigma, float* g_tint, float* g_diffuse, float* g_specular,
                       int gs_sigma, int gs_tint, int gs_diffuse, int gs_specular,
                       float* grad_rays_d, void* stream);

/* measurement hook: 1 = snrf_composite_fwd stages packed [R*S,10] head rows through shared memory as snrf_composite_bwd always
 * does (default 0: measured slower in the forward) */
void snrf_composite_set_fwd_packed(int on);
/* Early ray termination in TRAINING (opt-in; the north star's compositing subsystem.  The reference evaluates and
 * back-propagates every sample, hashgrid/__init__.py:512-596, so this is an approximation the caller chooses: ert_eps = 0
 * reproduces snrf_composite_fwd exactly).  A sample whose transmittance in front of it is below ert_eps is composited with
 * weight 0 and flagged dead in sample_live [R*S] (1 = live; 0 also for the samples of masked-out rays; may be NULL).  In the
 * joint batch (infinity != 0, R == 2 * inf_start: ray r + R/2 = the background chain of foreground ray r) the background
 * samples are tested against T_left(foreground) * T.  The *_ert backward entry points below take the flags and skip the dead
 * samples: zero head gradients (snrf_composite_bwd_ert), decoder tiles without a live sample skipped and grad_feats rows of
 * dead samples left unwritten (snrf_decoder_bwd_ert), no table / ray gradient from them (snrf_field_encode_bwd{,_adam}_ert). */
int snrf_composite_fwd_ert(const float* sigma, const float* tint, const float* diffuse, const float* specular,
                           int s_sigma, int s_tint, int s_diffuse, int s_specular,
                           const float* z_vals, const float* dists, const float* rays_d, const unsigned char* ray_valid,
                           int R, int S, int infinity, int inf_start, float* weights, float* trans, float* out,
                           float ert_eps, unsigned char* sample_live, void* stream);
int snrf_composite_bwd_ert(const float* sigma, const float* tint, const float* diffuse, const float* specular,
                           int s_sigma, int s_tint, int s_diffuse, int s_specular,
                           const float* z_vals, const float* dists, const float* rays_d, const float* trans,
                           const float* g_out, const float* g_weights, const unsigned char* ray_valid, int R, int S, int infinity,
                           int inf_start, float* g_sigma, float* g_tint, float* g_diffuse, float* g_specular,
                           int gs_sigma, int gs_tint, int gs_diffuse, int gs_specular,
                           float* grad_rays_d, const unsigned char* sample_live, void* stream);
int snrf_decoder_bwd_ert(const float* feats, const float* mask32, const float* rays_d, const float* const* params,
                         const float* grad_heads, float* grad_feats, float* grad_rays_d, float* const* grad_params,
                         int N, int S, int level_major, const unsigned char* ray_valid, const float* heads_fwd,
                         const unsigned char* sample_live, void* stream);
int snrf_field_encode_bwd_ert(const float* rays_o, const float* rays_d, const float* z_vals, const float* points,
                              const float* box_min, const float* box_size, int mode, const int* res, const float* grad_lm,
                              const float* jac_lm, float* grad_rays_o, float* grad_rays_d, float* grad_points, float* grad_table,
                              const unsigned char* ray_valid, int split, int N, int S, int L, int T,
                              const unsigned char* sample_live, void* stream);
int snrf_field_encode_bwd_adam_ert(const float* rays_o, const float* rays_d, const float* z_vals, const float* points,
                                   const float* box_min, const float* box_size, int mode, const int* res, const float* grad_lm,
                                   const float* jac_lm, float* grad_rays_o, float* grad_rays_d, float* grad_points,
                                   float* table, float* exp_avg, float* exp_avg_sq, float lr, float beta1, float beta2, float eps,
                                   int step, float* grad_scratch, long long scratch_entries, int small_levels, float* cpts_scratch,
                                   const unsigned char* ray_valid, int split, int N, int S, int L, int T,
                                   const unsigned char* sample_live, void* stream);

/* Colour loss of the joint foreground + background batch, value and gradient in one pass: replaces the torch chain between the
 * compositing rows and loss.backward() in TILE.train_one_step -- the merge of the two chains (tile.py:661-681), the clamp of
 * HashGrid.render_batch_rays (hashgrid/__init__.py:589), the masked MSE (criterions.py:126-147), the specular L2 regulariser
 * (tile.py:999).  row [2R,16] = rows of snrf_composite_fwd (rays [0,R) foreground, [R,2R) the background chains of the same
 * pixels); valid_f / valid_b [R] bytes; gt [R,3].
 *   pred = clamp(dif_f + spec_f, 0, 1) + T_left_f * clamp(dif_b + spec_b, 0, 1)
 *   loss = sum_{valid_f | valid_b} |pred - gt|^2 / (3 n_valid) + l2_weight * (sum row_f[10:13] / (3 n_f) + sum row_b[10:13] / (3 n_b))
 * loss: one float, ACCUMULATED (zero it first); g_row [2R,16] = d loss / d row, WRITTEN; pred_color [R,3] optional;
 * counts_scratch: 3 ints of device scratch. */
int snrf_joint_loss(const float* row, const unsigned char* valid_f, const unsigned char* valid_b, const float* gt,
                    float l2_weight, int R, float* loss, float* g_row, float* pred_color, int* counts_scratch, void* stream);

/* ---- decoder MLP on the tensor cores (tcgen05 / TMEM) ------------------------- */
/* Self-test of the tensor-core conventions (no reference counterpart): X[128,64], W[64,64],
 * G[128,64] f32, rounded to bf16 inside -> Y = X W^T [128,64], DX = G W [128,64],
 * DW = 2 G^T X [64,64], DWo = G^T X[:,32:48] [64,16], YS = X[:,32:64] W[0:16,0:32]^T [128,16] (f32). */
int snrf_umma_selftest(const float* X, const float* W, const float* G, float* Y, float* DX, float* DW,
                       float* DWo, float* YS, void* stream);

/* network.py:151-190 (ShallowMLP.forward): feats[N,32] f32 (hash-encode output), mask32[32] f32
 * (level mask, NULL = ones), rays_d[R,3] (sample n belongs to ray n / S; normalised inside with the
 * reference's +1e-8), params = HOST array of 16 DEVICE pointers in network.ShallowMLP state_dict
 * order (weight, bias per Linear: Spatial_MLP.mlp.0 [64,32], .mlp.2 [64,64], sigma_layer [1,32],
 * diffuse_layer [3,32], tint_layer [3,32], Directional_MLP.mlp.0 [64,48], .2 [64,64], .4 [3,64]).
 * -> heads[N,10] f32 = (sigma, tint3, diffuse3, specular3).  bf16(x3) operands, f32 accumulation.
 * level_major != 0: feats (and grad_feats in the backward) are [16][N] float2, the layout of snrf_field_encode_*.
 * ray_valid (optional, bytes [R]): samples of rays with a 0 flag are skipped (their output rows are left untouched). */
int snrf_decoder_fwd(const float* feats, const float* mask32, const float* rays_d, const float* const* params,
                     float* heads, int N, int S, int level_major, const unsigned char* ray_valid, void* stream);

/* Operand precision of the decoder GEMMs: 1 (default) = error-compensated bf16x3 split operands in
 * every forward GEMM (~fp32 accuracy), 0 = plain bf16 operands (fastest). */
void snrf_decoder_set_precision(int split);
/* Backward of snrf_decoder_fwd (autograd of network.py:151-190).  heads_fwd[N,10] (REQUIRED, non-NULL) = the heads
 * snrf_decoder_fwd returned for these inputs.  grad_heads[N,10] (column order of heads) -> grad_feats[N,32] WRITTEN;
 * grad_rays_d[R,3] ACCUMULATED (may be NULL; the view direction enters through the SH encoding only); grad_params = HOST
 * array of 16 DEVICE pointers, shapes/order of params, ACCUMULATED.  The forward is recomputed per 128-sample tile up to
 * layer 4, with layer 2 (linear, no activation) folded into its consumers. */
int snrf_decoder_bwd(const float* feats, const float* mask32, const float* rays_d, const float* const* params,
                     const float* grad_heads, float* grad_feats, float* grad_rays_d, float* const* grad_params,
                     int N, int S, int level_major, const unsigned char* ray_valid, const float* heads_fwd, void* stream);

/* ---- view selection, neighbour projection, image sampling ------------------------ */
/* cuda/include/view_selection.h (computeViewcost; kernel cuda/view_selection_kernel.cu:18-76):
 * rays_o, rays_d, pts [B,3]; ks [N,9]; rts [N,12] world->camera -> costs [N,B]. */
int snrf_view_cost(const float* rays_o, const float* rays_d, const float* pts, const float* ks, const float* rts,
                   float* costs, int n_cam, int B, int height, int width, void* stream);
/* proj2neighbor_forward (cuda/view_selection_kernel.cu:115-212): nei_views [B,K] i32, nei_valid [B,K] bytes
 * -> nei_origin, nei_direction, grid [B,K,3] (grid = K (R p + t), not dehomogenised); invalid pairs untouched. */
int snrf_proj2nei_fwd(const float* pts, const float* ks, const float* rts, const int* nei_views,
                      const unsigned char* nei_valid, float* nei_origin, float* nei_direction, float* grid, int B, int K,
                      void* stream);
/* proj2neighbor_backward (cuda/view_selection_kernel.cu:214-352): ACCUMULATES grad_pts [B,3], grad_rts [N,12]. */
int snrf_proj2nei_bwd(const float* pts, const float* ks, const float* rts, const int* nei_views,
                      const unsigned char* nei_valid, const float* dL_dgrid, float* grad_pts, float* grad_rts, int B, int K,
                      int n_cam, void* stream);
/* grid_sample_forward_cuda / grid_sample_backward_cuda (cuda/grid_sample_kernel.cu:109-213): src [N,H,W,3] u8,
 * grid [N,B,1,2] in [-1,1] (align-corners) -> out [N,B,1,3] f32, mask [N,B,1,1] bytes; grad_grid [N,B,1,2]. */
int snrf_grid_sample_fwd(const unsigned char* src, const float* grid, float* out, unsigned char* mask, int n_img, int B,
                         int height, int width, void* stream);
int snrf_grid_sample_bwd(const unsigned char* src, const float* grid, const float* grad_in, float* grad_grid, int n_img,
                         int B, int height, int width, void* stream);
/* gaussian_grid_sample_forward/backward_cuda (cuda/grid_sample_kernel.cu:216-441) */
int snrf_gauss_sample_fwd(const unsigned char* src, const float* grid, float* out, unsigned char* mask, int n_img, int B,
                          int height, int width, float sigma, float max_dis, void* stream);
int snrf_gauss_sample_bwd(const unsigned char* src, const float* grid, const float* grad_in, float* grad_grid, int n_img,
                          int B, int height, int width, float sigma, float max_dis, void* stream);
/* Neighbour-view colour fetch of the warp loss (warp_loss.py:441-519, WarpLoss.sample_neighbor_color; the reference
 * does this with host-resident images and four CPU gathers per step).  images [N,H,W,3] u8 resident on the device,
 * occlusion [N,H,W] bytes or NULL, grid [B,K,2] pixel coordinates, nei_views [B,K] i32, nei_valid [B,K] bytes ->
 * color [B,K,3] f32 in [0,1] (bilinear, taps clamped into the image), valid_out [B,K] = nei_valid & occlusion at the
 * nearest pixel.  The backward writes grad_grid [B,K,2] = d color / d grid contracted with grad_color. */
int snrf_nei_sample_fwd(const unsigned char* images, const unsigned char* occlusion, const float* grid, const int* nei_views,
                        const unsigned char* nei_valid, float* color, unsigned char* valid_out, int B, int K, int height,
                        int width, void* stream);
int snrf_nei_sample_bwd(const unsigned char* images, const float* grid, const int* nei_views, const unsigned char* nei_valid,
                        const float* grad_color, float* grad_grid, int B, int K, int height, int width, void* stream);
/* grid_sample_bool_cuda (cuda/grid_sample_kernel.cu:445-493): src [N,H,W] bytes; out-of-image entries keep their value */
int snrf_grid_sample_bool(const unsigned char* src, const float* grid, unsigned char* out, int n_img, int B, int height,
                          int width, void* stream);
/* proj2pixel_and_fetch_color (cuda/helper_kernel.cu:17-104): C2Ws [N,12] camera->world, rgbs [N,H,W,3] f32
 * -> fetched_pixels, fetched_colors [B,N,3]. */
int snrf_proj2pixel_fetch(const float* pts, const float* Ks, const float* C2Ws, const float* rgbs, float* fetched_pixels,
                          float* fetched_colors, int B, int n_cam, int height, int width, void* stream);

/* ---- multi-tile inference renderer (hashgrid/include/rendering.h:20-182) --------- */
/* "block" = tile.  corners/sizes [nb,3]; grid_occupied = concatenated byte grids, grid_starts [nb] i64,
 * grid_log2dim [nb,3] i32; intersections [B,nb,2] (1e7 = miss); tracing_blocks [B,nb] i32 = tiles near-to-far. */
int snrf_ray_block_isect(const float* rays_o, const float* rays_d, const float* corners, const float* sizes,
                         float* intersections, int B, int nb, void* stream);                         /* ray_block_intersection */
int snrf_render_sample(const float* rays_o, const float* rays_d, const float* corners, const float* sizes,
                       const unsigned char* grid_occupied, const long long* grid_starts, const int* grid_log2dim,
                       const int* tracing_blocks, const float* intersections, int* tracing_idx, float* z_start,
                       float* z_vals, float* dists, int B, int nb, int S, void* stream);             /* sample_points */
int snrf_prepare_points(const float* z_vals, const unsigned char* running_mask, const float* intersections,
                        short* block_idxs, int B, int S, int nb, void* stream);                      /* prepare_points */
int snrf_accumulate(const float* pts_diffuse, const float* pts_specular, const float* pts_alpha, float* transparency,
                    const float* z_vals, float* diffuse, float* specular, float* depth, int B, int S, void* stream); /* accumulate_color */
int snrf_ray_firsthit_block(const float* rays_o, const float* rays_d, const float* corners, const float* sizes,
                            const unsigned char* grid_occupied, const long long* grid_starts, const int* grid_log2dim,
                            const int* tracing_blocks, const float* intersections, short* hit_block_idxs, int B, int nb,
                            void* stream);                                                            /* ray_firsthit_block */
int snrf_inverse_z(const float* intersections, const short* related_bidx, float* z_vals, float sample_range, int B,
                   int nb, int S, void* stream);                                                      /* inverse_z_sampling */
int snrf_get_last_block(const int* tracing_blocks, int* bidxs, const float* intersections, int B, int nb, void* stream);
int snrf_outgoing_bidx(const float* rays_o, const float* rays_d, const float* corners, const float* sizes,
                       const int* tracing_blocks, const float* intersections, short* outgoing_bidxs, float* blend_weights,
                       int skip, int B, int nb, void* stream);                                        /* update_outgoing_bidx */
int snrf_inside_bidx(const float* rays_o, const float* corners, const float* sizes, short* inside_bidxs,
                     float* blend_weights, int B, int nb, void* stream);                              /* update_outgoing_bidx_v2 */
int snrf_process_occupied(int bidx, int total_grid, const float* corners, const float* sizes,
                          const unsigned char* grid_occupied, const long long* grid_starts, const int* grid_log2dim,
                          unsigned char* tgt_grid_occupied, int nb, void* stream);                    /* process_occupied_grid */
/* Fused fp16-table encode + decoder MLP (tensor cores) + alpha + overlap blending.
 * features_tables [nb,16,T,2] f16; params [nb,13994] f32 in the renderer's flat layout (rendering.py:101-113);
 * resolution [nb,16,3] i32; nb = number of tiles.  pts_inference: block_idxs [B,S,4] i16, outputs [B,S,3],[B,S,3],[B,S,1]. */
int snrf_pts_inference(const float* rays_o, const float* rays_d, const float* z_vals, const float* dists,
                       const short* block_idxs, const void* features_tables, const float* params, const int* resolution,
                       const unsigned char* grid_occupied, const long long* grid_starts, const int* grid_log2dim,
                       const float* corners, const float* sizes, float* diffuse, float* specular, float* alpha, int B,
                       int S, int T, int nb, void* stream);
int snrf_bg_pts_inference(const float* rays_o, const float* rays_d, const float* z_vals, const short* outgoing_bidxs,
                          const float* blend_weights, const float* corners, const float* sizes, const int* resolution,
                          const void* features_tables, const float* params, float* diffuse, float* specular, float* alpha,
                          int B, int S, int T, int nb, void* stream);
int snrf_bg_pts_inference_v2(const float* rays_o, const float* rays_d, const float* z_vals, const short* bg_idxs, int step,
                             const float* corners, const float* sizes, const int* resolution, const void* features_tables,
                             const float* params, float* diffuse, float* specular, float* alpha, int B, int S, int T,
                             int nb, void* stream);
/* tuning hook: log2 of the samples per chunk of the single-tile two-pass evaluation behind pts_inference / bg_pts_inference*
 * (20 .. 26): a chunk streams the table from HBM once, its scratch is 153 B per sample */
void snrf_infer_set_chunk_log2(int bits);
/* The multi-pass inference paths keep their scratch (features of one 4 Mi-sample chunk, <= 3.1 GB) in a private
 * stream-ordered pool between calls; this synchronises the device and returns that memory to the driver. */
int snrf_infer_release_scratch(void);

/* ---- sparse Adam -------------------------------------------------------------- */
/* cuda/include/adam.h (adam_step_cuda: half_state=0, adam_step_cuda_fp16: half_state=1; kernels
 * cuda/adam_kernel.cu:23-69, 97-144).  Element (k,d), k<rows, d<dim, lives at k*row_stride+d
 * (the reference hard-codes row_stride 8).  Elements whose gradient is exactly 0 are skipped.
 * exp_avg / exp_avg_sq are f32 (half_state=0) or f16 scaled by 128 / 128^2 (half_state=1).
 * `step` is the 1-based step used in the bias corrections (the reference passes step+1).
 * zero_grad != 0 clears every consumed gradient in the same pass (extension). */
int snrf_adam_step(float* params, float* grads, void* exp_avg, void* exp_avg_sq,
                   long long rows, int dim, int row_stride, int half_state,
                   float lr, float beta1, float beta2, float eps, int step, int zero_grad,
                   void* stream);

/* ---- image-quality metrics ---------------------------------------------------------- */
/* tile.py:810-864 / rendering.py val mode score held-out views on the host (tools/ssim.py); here on the device.
 * pred[N,H,W,3] f32; gt[N,H,W,3] u8 (gt_is_u8=1, read as (float)v / 255.0f) or f32 (gt_is_u8=0);
 * mask[N,H,W] bytes, non-zero = score the pixel (NULL = every pixel).
 * -> out_mse[N], out_ssim[N]: means over the masked pixels and the 3 channels (NaN when no pixel is masked in),
 *    out_count[N]: masked pixels.  SSIM: 11x11 Gaussian window (sigma 1.5), zero padding, C1 = 0.01^2, C2 = 0.03^2
 *    (pytorch-ssim; the mask selects map values, it does not change the local statistics).
 * scratch: N * ceil(H/16) * ceil(W/32) * 3 doubles of device memory.  Deterministic: the same inputs give the same bits. */
int snrf_image_metrics(const float* pred, const void* gt, int gt_is_u8, const unsigned char* mask, int N, int H, int W,
                       float* out_mse, float* out_ssim, float* out_count, void* scratch, size_t scratch_bytes, void* stream);

/* ---- ray <-> proxy mesh (fastMesh) --------------------------------------------- */
/* fastMesh/include/fastMesh.h:11-57 (class fastMesh).  The handle owns one device allocation on
 * the current device; queries may run on any stream of that device. */
int snrf_mesh_create(const char* ply_path, void** handle);                 /* build(path): fastMesh.h:22-26 */
int snrf_mesh_create_from_arrays(const float* verts_host, int nv, const int* faces_host, int nf, void** handle);
int snrf_mesh_destroy(void* handle);                                        /* destroy(): fastMesh.h:52-55 */
int snrf_mesh_bounds(void* handle, float* bound6_host);                     /* getSceneBound(): fastMesh.h:28-38 */
int snrf_mesh_stats(void* handle, long long* stats3_host);                  /* occupied cells, list entries, faces */
/* fisrtHit (sic) fastMesh_kernel.cu:230-329: z_depth[B] = nearest t>0 within the first cell that has a
 * hit, 0 = miss; hit_face[B] i32 optional (extension): that face's index or -1. */
int snrf_mesh_first_hit(void* handle, const float* rays_o, const float* rays_d, float* z_depth, int* hit_face,
                        int B, void* stream);
/* firstEnter fastMesh_kernel.cu:125-227 */
int snrf_mesh_first_enter(void* handle, const float* rays_o, const float* rays_d, float* z_depth, int B, void* stream);
/* sample_points fastMesh_kernel.cu:23-122: t_start[B] (-1 = leave the row untouched), z_vals[B,S] */
int snrf_mesh_sample(void* handle, const float* rays_o, const float* rays_d, const float* t_start, float* z_vals,
                     int B, int S, void* stream);

/* ---- mesh ingest (host) ------------------------------------------------------- */
/* cuda/include/voxelize.h:12-119 (voxelize_mesh): ALL pointers are host pointers.
 * log2dim[3], corner[3], size[3]; vis / outside: bytes [2^lx * 2^ly * 2^lz]. */
int snrf_voxelize_mesh_host(const int* log2dim, const float* corner, const float* size,
                            const char* model_path, unsigned char* vis, int init_out,
                            unsigned char* outside);

#ifdef __cplusplus
}
#endif
#endif /* SCANERF_B200_H */
