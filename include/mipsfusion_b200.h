/* mipsfusion_b200 -- C ABI of the B200-native MIPSFusion per-frame neural-field hot path.
 *
 * This is the drop-in boundary (SURVEY.md 8b).  The reference has no C ABI: its
 * boundary is Python (tcnn.Encoding, MLP_reg, JointEncoding, RandomOptimizer,
 * Mesher).  Each entry point below names the reference interface it replaces
 * (file:line relative to the reference checkout); the Python host mirror in
 * mipsfusion_b200/ binds them with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - tensors are dense row-major fp32 unless stated; sizes are element counts;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and
 *     nothing synchronises the device;
 *   - return value: 0 on success, negative on error (MF_ERR_*); the message is
 *     retrievable with mf_last_error() (thread-local).  Nothing throws or aborts;
 *   - no global mutable state besides a per-process cache of device attributes.
 */
#ifndef MIPSFUSION_B200_H
#define MIPSFUSION_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MF_ABI_VERSION 2
#define MF_MAX_LEVELS 16
#define MF_MLP_PARAMS 36577          /* reference model/decoder.py:32-50 with input_ch=32, input_ch_pos=48 */
#define MF_RAW_DIM 10                /* rgb_raw(3) sdf(1) entropy(1) prob(5), model/decoder.py:74 */

#define MF_OK 0
#define MF_ERR_INVALID (-1)
#define MF_ERR_CUDA (-2)
#define MF_ERR_UNSUPPORTED (-3)

/* Per-level table of the multi-resolution hash grid (tinycudann 1.7 GridEncoding;
 * reference model/encodings.py:11-26).  Host-side POD, filled by mf_hashgrid_meta. */
typedef struct {
    int32_t n_levels, n_features, log2_hashmap_size, base_resolution;
    float scale[MF_MAX_LEVELS];
    uint32_t resolution[MF_MAX_LEVELS];
    uint32_t size[MF_MAX_LEVELS];          /* entries per level */
    uint32_t offset[MF_MAX_LEVELS + 1];    /* entry offsets; offset[n_levels] = total entries */
    uint32_t hashed[MF_MAX_LEVELS];        /* 1: coherent-prime hash, 0: dense stride index */
} mf_grid_meta;

/* One submap's neural field ("localMLP"): reference model/scene_rep.py:11-45.
 * Coordinate normalisation (scene_rep.py:138-142) is x_n = ((double)x - norm_a) / norm_b
 * / norm_factor, evaluated in fp64 and rounded to fp32 once, as in the reference.
 *   use_bound_normalize: norm_a = bound_min, norm_b = bound_max - bound_min
 *   otherwise:           norm_a = -L,        norm_b = 2 L          (L = localMLP_max_len) */
typedef struct {
    const float* grid;        /* embed_fn.params, flat fp32, n_params */
    const float* mlp_prep;    /* kernel-layout weights written by mf_mlp_prepare */
    double norm_a[3], norm_b[3];
    double norm_factor;       /* training.norm_factor */
    int32_t decoder_impl;     /* 0: process default (mf_set_decoder_impl), 1: fp32 CUDA cores, 2: tcgen05 tensor cores */
    int32_t reserved;
    mf_grid_meta meta;
} mf_field;

/* Scalars of reference model/scene_rep.py:153-238 + helper_functions/utils.py. */
typedef struct {
    int32_t n_samples_d;      /* training.n_samples_d (uniform); or training.n_samples when target_d is NULL */
    int32_t n_range_d;        /* training.n_range_d (around depth); 0 when target_d is NULL */
    int32_t perturb;          /* training.perturb > 0 */
    int32_t rgb_missing_nz;   /* training.rgb_missing != 0 */
    double trunc;             /* training.trunc        (python floats are doubles; the kernels round */
    double sc_factor;         /* data.sc_factor         them to fp32 exactly where torch would)      */
    double depth_trunc;       /* cam.depth_trunc */
    double emd_w;             /* EMD_w argument of JointEncoding.forward */
} mf_render_cfg;

const char* mf_last_error(void);
int mf_abi_version(void);
/* Number of SMs of the current device (grid sizing); <0 on error. */
int mf_device_sm_count(void);

/* Decoder implementation used by the forward field kernels: 0 = tcgen05 tensor cores with a bf16x3 split
 * (default), 1 = fp32 CUDA cores (numerical reference).  Process-wide; meant for verification. */
int mf_set_decoder_impl(int impl);
int mf_get_decoder_impl(void);
/* 1 if a tensor-core kernel reported an MMA-completion timeout since the last call (clears the flag;
 * synchronises the device -- diagnostics only). */
/* A/B switch of the tensor-core backward: 0 = three-role kernel (default), 1 = single-role kernel of round 1, 3 = four-role kernel (A/B only). */
int mf_set_bwd_impl(int impl);
/* A/B switch of the forward kernel's tile scheduling: 1 = dynamic (global tile counter, default), 0 = static striding. */
int mf_set_dynamic_tiles(int on);
/* Number of SMs the forward kernel leaves free (default 0).  The data-parallel mapper sets 1 so that its count all-reduce, issued
 * on the collective library's stream, overlaps the forward instead of waiting for an SM. */
int mf_set_sm_reserve(int n);
int mf_tc_check_error(void);
/* Diagnostics: out (128,128) = x (128,K) w (128,K)^T through one tcgen05 layer; K % 16 == 0, K <= 128;
 * passes = 1 (bf16) or 3 (bf16x3 split). */
int mf_debug_umma_linear(const float* x, const float* w, float* out, int K, int passes, void* stream);
/* Diagnostics: out (128,Kf) = dz (128,128) w (128,Kf)  (dgrad data path: TMEM A, MN-major weight image), Kf in {64,96,128}. */
int mf_debug_umma_dgrad(const float* dz, const float* w, float* out, int Kf, void* stream);
/* Diagnostics: out (128,Kf)[n][k] = sum_p dz[p][n] x[p][k] over 128 points (wgrad data path: both operands MN-major
 * from shared memory, two 64-point half tiles); passes = 1 (dz_hi x_hi) or 2 (+ dz_lo x_hi). */
int mf_debug_umma_wgrad(const float* dz, const float* x, float* out, int Kf, int passes, void* stream);

/* Diagnostics: switch the in-kernel clock stamps of the tensor-core backward on/off and read the last ones. */
int mf_debug_profile(int on, long long* out_host);
/* All stamps (n <= 1024 int64): [0,64) as above; [64+2b, 65+2b] / [576+2b, 577+2b] = %globaltimer (ns) at the start / end of
 * CTA b of the last profiled forward / backward tensor-core kernel.  Diagnostics only. */
int mf_debug_profile_all(long long* out_host, int n);
/* Diagnostics for bench.py's roofline line: when on, the launchers bracket the dominant kernel itself with a CUDA event pair
 * on the launching stream (slot 0 field forward, 1 field backward, 2 RandomOptimizer field query, 3 joint-query field query);
 * mf_debug_kernel_ms waits for the last bracketed launch of `slot` and returns its duration. */
int mf_debug_kernel_timer(int on);
int mf_debug_kernel_ms(int slot, float* ms);

/* ---- a1: hash-grid encoding (replaces tcnn.Encoding "HashGrid", model/encodings.py:14-25) ---- */
int mf_hashgrid_meta(int log2_hashmap_size, int n_levels, int n_features, int base_resolution,
                     double per_level_scale, mf_grid_meta* meta_host);
/* x (N,3) in the unit cube (wraps outside) -> out (N, L*F).  idx_dump (N,L,8) uint32 optional (NULL). */
int mf_hashgrid_fwd(const float* x, const float* grid, const mf_grid_meta* meta_host, float* out,
                    uint32_t* idx_dump, int64_t N, void* stream);
/* grad_grid += scatter(dL_dy); dL_dx (N,3) optional (NULL). */
int mf_hashgrid_bwd(const float* x, const float* dL_dy, const float* grid, const mf_grid_meta* meta_host,
                    float* grad_grid, float* dL_dx, int64_t N, void* stream);

/* ---- a2: frequency encoding (replaces tcnn.Encoding "Frequency", model/encodings.py:31-38) ---- */
int mf_freq_fwd(const float* x, float* out, int n_dims, int n_frequencies, int64_t N, void* stream);
int mf_freq_bwd(const float* x, const float* dL_dy, float* dL_dx, int n_dims, int n_frequencies, int64_t N, void* stream);

/* ---- a3: decoder MLP_reg (model/decoder.py:6-75) ---- */
/* `mlp` is the flat concatenation of the state_dict tensors in order:
 * pts_linear.0.{weight(128,51),bias} pts_linear.2.{(128,128),bias} rgb_linear.0.{(3,115),bias}
 * sdf_linear.0.{(128,96),bias} sdf_linear.2.{(5,128),bias}  = MF_MLP_PARAMS floats.
 * mf_mlp_prepare re-lays it out for the kernels into mlp_prep (mf_mlp_prep_size() floats). */
int64_t mf_mlp_prep_size(void);
int mf_mlp_prepare(const float* mlp, float* mlp_prep, void* stream);
/* MLP_reg.forward(embed (N,32), embed_pos (N,48), query_pts (N,3)) -> out (N,10) */
int mf_mlp_fwd(const float* embed, const float* embed_pos, const float* pts, const float* mlp_prep,
               float* out, int64_t N, void* stream);
/* grad_mlp (MF_MLP_PARAMS, same layout as `mlp`) += ...; d_embed/d_embed_pos/d_pts optional (NULL).
 * workspace: mf_mlp_grad_workspace_size() floats of scratch (per-CTA partial sums). */
int64_t mf_mlp_grad_workspace_size(void);
int mf_mlp_bwd(const float* embed, const float* embed_pos, const float* pts, const float* mlp_prep,
               const float* d_out, float* grad_mlp, float* d_embed, float* d_embed_pos, float* d_pts,
               float* workspace, int64_t N, void* stream);

/* ---- a4: fused field query (JointEncoding.run_network / query_*, model/scene_rep.py:106-146) ----
 * pts (N,3) fp32 in the submap frame -> out (N,10).  normalize=0 skips the bound normalisation
 * (query_color_sdf called directly on pre-normalised points, as model/Mesher.py:487 does). */
int mf_field_query(const float* pts, const mf_field* field_host, int normalize, float* out, int64_t N, void* stream);
/* backward of the above: grad_grid/grad_mlp accumulate; d_pts (N,3) optional.  grad_grid = grad_mlp = NULL: point gradients
 * only (d_pts required; no weight gradients, no grid scatter; fp32 or tensor-core decoder as the field selects).
 * workspace: mf_field_bwd_workspace_size(N, 0) floats (per-CTA partial sums + the list of points whose d_out row is
 * non-zero: rows that are exactly zero add nothing to any gradient and are skipped). */
int64_t mf_field_bwd_workspace_size(int64_t n_points, int want_ray_grads);
int mf_field_query_bwd(const float* pts, const mf_field* field_host, int normalize, const float* d_out,
                       float* grad_grid, float* grad_mlp, float* d_pts, float* workspace, int64_t N, void* stream);

/* ---- a5: z sampling (JointEncoding.render_rays, model/scene_rep.py:157-176) ----
 * target_d (R) or NULL; u (R,S) jitter in [0,1) (the reference's torch.rand) or NULL when perturb=0;
 * lin_uniform (n_samples_d) = linspace(near, far, n_samples_d); lin_range (n_range_d) =
 * linspace(-range_d, range_d, n_range_d); lin_fallback (n_range_d) = linspace(near, far, n_range_d).
 * Writes z (R,S), S = n_samples_d + n_range_d, and the global mask counts
 * counts[0] = #front samples, counts[1] = #sdf samples (helper_functions/utils.py:43-44; int64, zeroed here). */
int mf_sample_z(const float* target_d, const float* u, const float* lin_uniform, const float* lin_range,
                const float* lin_fallback, const mf_render_cfg* cfg_host, float* z, int64_t* counts,
                int64_t R, void* stream);

/* ---- a4+a12 fused: points on rays pts = o + d z, field query -> raw (R,S,10) ---- */
/* feat (optional, NULL to skip): cache of the encoded features, mf_feat_cache_size(R*S) bytes, written by the
 * forward and consumed by mf_field_query_rays_bwd so that the backward does not repeat the table gathers
 * (tensor-core decoder only; ignored by the fp32 decoder). */
int64_t mf_feat_cache_size(int64_t n_points);
int mf_field_query_rays(const float* rays_o, const float* rays_d, const float* z, const mf_field* field_host,
                        float* raw, void* feat, int64_t R, int S, void* stream);
/* d_raw (R,S,10) -> grad_grid, grad_mlp (accumulate), d_rays_o / d_rays_d (R,3; optional, overwritten).
 * grad_grid == grad_mlp == NULL with d_rays_o / d_rays_d given: ray gradients only (the gradient pose refinement of tracking,
 * mipsfusion.py:501-556, needs nothing else; tensor-core decoder).
 * workspace: mf_field_bwd_workspace_size(R*S, d_rays_o != NULL) floats. */
int mf_field_query_rays_bwd(const float* rays_o, const float* rays_d, const float* z, const mf_field* field_host,
                            const float* d_raw, const void* feat, float* grad_grid, float* grad_mlp, float* d_rays_o,
                            float* d_rays_d, float* workspace, int64_t R, int S, void* stream);

/* ---- a6-a8: SDF->weights rendering + losses (scene_rep.py:58-103,190-238; helper_functions/utils.py:21-111) ----
 * out_rgb (R,3), out_depth (R), out_aux (R,3) = depth_var, disp_map, acc_map (optional); out_weights (R,S) normalised
 * sample weights (optional); inds (R) int32 first-sign-change index (optional);
 * losses (8) = rgb_loss, depth_loss, sdf_loss, fs_loss, psnr, fs_weight, sdf_weight, n_valid.
 * target_rgb/target_d NULL => render only (eval mode), losses untouched.  scratch: R*8 floats. */
int mf_render_loss_fwd(const float* raw, const float* z, const float* target_rgb, const float* target_d,
                       const int64_t* counts, const mf_render_cfg* cfg_host, float* out_rgb, float* out_depth,
                       float* out_aux, float* out_weights, int32_t* inds, float* losses, float* scratch,
                       int64_t R, int S, void* stream);
/* _ld variants: target_rgb / target_d are R rows with row strides ld_rgb >= 3 / ld_d >= 1 floats -- the column slices the
 * reference's loop takes out of its (R,10) batch tensor (mipsfusion.py:316-322) are read in place, without a copy each. */
int mf_sample_z_ld(const float* target_d, int ld_d, const float* u, const float* lin_uniform, const float* lin_range,
                   const float* lin_fallback, const mf_render_cfg* cfg_host, float* z, int64_t* counts, int64_t R, void* stream);
int mf_render_loss_fwd_ld(const float* raw, const float* z, const float* target_rgb, int ld_rgb, const float* target_d, int ld_d,
                          const int64_t* counts, const mf_render_cfg* cfg_host, float* out_rgb, float* out_depth,
                          float* out_aux, float* out_weights, int32_t* inds, float* losses, float* scratch,
                          int64_t R, int S, void* stream);
/* g_losses (4) upstream grads of rgb/depth/sdf/fs loss (device); g_rgb (R,3) / g_depth (R) optional upstream
 * grads of the rendered maps -> d_raw (R,S,10). */
int mf_render_loss_bwd(const float* raw, const float* z, const float* target_rgb, const float* target_d,
                       const int64_t* counts, const float* losses, const mf_render_cfg* cfg_host,
                       const float* g_losses, const float* g_rgb, const float* g_depth, float* d_raw,
                       int64_t R, int S, void* stream);
/* The same with the four loss gradients as separate device scalars (NULL = 0): what autograd hands to the backward of a weighted
 * sum of the four losses (mipsfusion.py:142-152), without packing them first; target row strides as in the _ld variants below. */
int mf_render_loss_bwd_scalars(const float* raw, const float* z, const float* target_rgb, int ld_rgb, const float* target_d, int ld_d,
                               const float* losses, const mf_render_cfg* cfg_host, const float* g_rgb_loss, const float* g_depth_loss,
                               const float* g_sdf_loss, const float* g_fs_loss, const float* g_rgb, const float* g_depth,
                               float* d_raw, int64_t R, int S, void* stream);

/* ---- a10: dense Adam (torch.optim.Adam as configured at mipsfusion.py:580-584) ----
 * step >= 1; zero_grad != 0 also clears g (the reference's zero_grad, mipsfusion.py:335). */
int mf_adam_step(float* p, float* g, float* m, float* v, int64_t n, double lr, double beta1, double beta2,
                 double eps, double weight_decay, int step, int zero_grad, void* stream);

/* Data-parallel mapping (one process per GPU): gradient reduce-scatter + Adam + parameter all-gather in one kernel over
 * NVLink peer memory.  peer_bases (HOST array, `world` entries) = base address of every rank's arena in this process'
 * address space (symmetric / peer-mapped memory, identical layout on all ranks); off_p / off_g / off_g_clear = float
 * offsets of the parameters, of the gradient to reduce and of the gradient buffer to zero (-1: none) inside the arena.
 * Rank r updates slab r of the n parameters (n % 4 == 0) with its local moments m, v (full-size arrays, only the slab
 * is touched) from the rank-ordered mean of all ranks' gradients and stores the result into every rank's parameters.
 * multicast_base: address of the NVSwitch multicast mapping of the same arena (NVLS), or 0: with it the gradient sum is one
 * multimem.ld_reduce (reduced in the switch) and the parameter broadcast one multimem.st.
 * The caller issues a cross-GPU barrier before (all gradients complete) and after (all slabs delivered) the call. */
int mf_adam_step_sharded(const uint64_t* peer_bases, int world, int rank, int64_t off_p, int64_t off_g, int64_t off_g_clear,
                         float* m, float* v, int64_t n, double lr, double beta1, double beta2, double eps,
                         double weight_decay, int step, uint64_t multicast_base, void* stream);
/* The two Adam groups of a mapping step (mipsfusion.py:580-584: hash grid and decoder, each with its own lr / eps / weight
 * decay) in one launch, gradients cleared.  n0, n1 multiples of 4, 16-byte aligned arrays (pad the decoder blob with zeros:
 * a zero parameter with a zero gradient stays zero). */
int mf_adam_step_pair(float* p0, float* g0, float* m0, float* v0, int64_t n0, double lr0, double eps0, double wd0,
                      float* p1, float* g1, float* m1, float* v1, int64_t n1, double lr1, double eps1, double wd1,
                      double beta1, double beta2, int step, void* stream);
/* The same update for a parameter group of n_tensors tensors (host arrays of device pointers and sizes). */
int mf_adam_step_multi(int n_tensors, float* const* p_host, float* const* g_host, float* const* m_host,
                       float* const* v_host, const int64_t* n_host, double lr, double beta1, double beta2, double eps,
                       double weight_decay, int step, int zero_grad, void* stream);

/* ---- N3: submap containment tests of the Manager (Manager.py:159-244; helper_functions/geometry_helper.py:193-203) ----
 * n points -- either `pts` (n,3) as given, or the surface points t + (R dirs_cam[i]) * depth[i] of a frame with camera-to-world
 * pose `pose_c2w` (16 floats, row major, device), formed in the reference's fp32 operation order -- against k axis-aligned boxes
 * (xyz_min / xyz_max (k,3)), strict comparisons as pts_in_bbox.  cross != 0: every direction is paired with every depth (n * n
 * points, direction-major) -- what the broadcast of Manager.py:174 ((P,1,3) * (P,1)) actually evaluates in
 * find_highest_containing_ratio; compute_containing_ratio (:214) pairs them one to one (cross = 0).
 * mask (points,k) uint8 and / or counts (2k+1) int64: [0,k) points inside box j, [k,2k) points inside box j whose depth is > 0,
 * [2k] points with depth > 0 (pts: all valid). */
int mf_containment(const float* dirs_cam, const float* depth, const float* pose_c2w, const float* pts, const float* xyz_min,
                   const float* xyz_max, int k, int64_t n, int cross, uint8_t* mask, int64_t* counts, void* stream);

/* ---- a11: pixel samplers (helper_functions/sampling_helper.py:7-68), int64 outputs ---- */
int mf_sample_pixels_uniform(int img_h, int img_w, int num_h, int num_w, int64_t* rows, int64_t* cols, void* stream);
/* top-`num` of keys*mask(depth>0 [and not on the lattice]) by (value desc, index asc); keys (H*W) >= 0.
 * lattice_h/w = 0 => sample_valid_pixels_random (indices only, rows/cols may be NULL);
 * else sample_pixels_mix: rows/cols (num) = lattice then random.  workspace: mf_topk_workspace_size(H*W) bytes. */
int64_t mf_topk_workspace_size(int64_t n);
int mf_sample_pixels_topk(const float* depth, const float* keys, int img_h, int img_w, int lattice_h, int lattice_w,
                          int num, int64_t* indices, int64_t* rows, int64_t* cols, void* workspace, void* stream);

/* ---- a12: ray generation (mipsfusion.py:320-322; geometry_helper.py:107-123; datasets/utils.py:29) ----
 * dirs_cam (R,3); poses (K,4,4) c2w; pose_idx (R) int64 or NULL (=> pose 0) -> rays_o, rays_d (R,3). */
int mf_gen_rays(const float* dirs_cam, const float* poses, const int64_t* pose_idx, float* rays_o, float* rays_d,
                int64_t R, int K, void* stream);
/* The same on the packed host batch of the mapping loop (mipsfusion.py:289-290,310-322): rays7 (R,7) =
 * [dir_cam | rgb | depth] -> rays_o, rays_d, target_rgb (R,3), target_d (R). */
int mf_gen_rays_packed(const float* rays7, const float* poses, const int64_t* pose_idx, float* rays_o, float* rays_d,
                       float* target_rgb, float* target_d, int64_t R, int K, void* stream);
/* d_poses (K,4,4) += backward of mf_gen_rays (rotation block and translation column). */
int mf_gen_rays_bwd(const float* dirs_cam, const int64_t* pose_idx, const float* d_rays_o, const float* d_rays_d,
                    float* d_poses, int64_t R, int K, void* stream);
/* The same for the packed batch of mf_gen_rays_packed: the camera directions are the first 3 of the 7 floats of a ray record
 * (mipsfusion.py:289-290).  This is the pose-gradient leg of the mapping loop's backward (mipsfusion.py:275-282,338-342). */
int mf_gen_rays_packed_bwd(const float* rays7, const int64_t* pose_idx, const float* d_rays_o, const float* d_rays_d,
                           float* d_poses, int64_t R, int K, void* stream);

/* ---- N1 (first "next" row of SURVEY 8): keyframe ray store on the device (model/keyframeSet.py:25,76-79,170-175,386-437) ----
 * mf_kf_store: add_keyframe -- store_slot (n_rays,7) = [dir_cam | rgb | depth] of the pixels (rows[j], cols[j]) of a
 * full-resolution frame (dirs_cam (H*W,3), rgb (H*W,3), depth (H*W)); rows / cols = the uniform lattice (mf_sample_pixels_uniform). */
int mf_kf_store(const float* dirs_cam, const float* rgb, const float* depth, const int64_t* rows, const int64_t* cols,
                int img_w, int64_t n_rays, float* store_slot, void* stream);
/* sample_rays_in_submap for given index draws (the reference's random.sample results, here device int64 arrays):
 * store (num_kf, n_rays, 7); first / last keyframe ids, other_kf_ids (the related keyframes between them);
 * out_rays7 (n,7), out_kf_ids (n), out_kf_indices (n) with n = n_first + n_other + n_last, in the reference's order. */
int mf_kf_gather_rays(const float* store, int64_t n_rays, int64_t first_kf_id, const int64_t* other_kf_ids,
                      int64_t last_kf_id, int n_related, const int64_t* idx_first, int64_t n_first,
                      const int64_t* idx_other, int64_t n_other, const int64_t* idx_last, int64_t n_last,
                      float* out_rays7, int64_t* out_kf_ids, int64_t* out_kf_indices, void* stream);

/* Sampling without replacement on the device (the reference's python random.sample(range(n), k)): out[j] = perm(j), perm a
 * keyed pseudo-random permutation of [0, n) (4-round Feistel network + cycle walking; oracle/keyframes.py restates it). */
int mf_sample_distinct(int64_t n, int64_t k, uint32_t seed, int64_t* out, void* stream);
/* sample_rays_in_submap with the draws made inside the kernel (segment seeds seed, seed+1, seed+2 for the first / other /
 * latest keyframes); out_idx (optional) receives the drawn indices, the other outputs are as mf_kf_gather_rays. */
int mf_kf_sample_rays(const float* store, int64_t n_rays, int64_t first_kf_id, const int64_t* other_kf_ids, int64_t n_other_kf,
                      int64_t last_kf_id, int n_related, int64_t n_first, int64_t n_other, int64_t n_last, uint32_t seed,
                      float* out_rays7, int64_t* out_kf_ids, int64_t* out_kf_indices, int64_t* out_idx, void* stream);
/* The mapping batch of submap initialisation (first_frame_mapping / initialize_new_localMLP, mipsfusion.py:135-138,178,209):
 * ray j takes pixel index i = idx[j] (idx given; each in [0, H*W)) or i = perm(j) of the mf_sample_distinct permutation of
 * [0, H*W) with `seed` (idx NULL: the reference's random.sample(range(H*W), n)), decoded column-major h = i % H, w = i / H;
 * out_rays7 (n,7) = [dir_cam | rgb | depth] of pixel (h, w) of the frame (dirs_cam (H*W,3), rgb (H*W,3), depth (H*W),
 * row-major).  out_idx (optional, n) receives i.  0 <= n <= H*W; n = 0 is a no-op. */
int mf_frame_sample_rays(const float* dirs_cam, const float* rgb, const float* depth, int img_h, int img_w, int64_t n,
                         uint32_t seed, const int64_t* idx, float* out_rays7, int64_t* out_idx, void* stream);

/* ---- gradient pose refinement of tracking (mipsfusion.py:501-556; get_pose_param_optim :235-241, qt_to_transform_matrix
 * geometry_helper.py:11-17) on the device.  state (32 floats): [0:4] quaternion (w,x,y,z), [4:7] translation, [7:14] Adam m,
 * [14:21] Adam v, [21] step count, [22] best loss (< 0: none yet), [23] iterations since the best (thresh), [24] stopped flag,
 * [25:32] spare.  best_c2w (16 floats) follows the reference: the pose whose loss was the smallest so far.
 * mf_pose_to_c2w: state -> c2w (4,4), pytorch3d quaternion_to_matrix (no unit-norm assumption). */
int mf_pose_to_c2w(const float* state, float* c2w, void* stream);
/* One refinement update: losses (>= 4 floats: rgb, depth, sdf, fs) and loss_w (4) give the scalar the reference compares;
 * best / thresh / stopped are updated exactly as the loop body does (:540-552); unless stopped, d_c2w (4,4) is pulled back to the
 * quaternion and the translation and one torch.optim.Adam step (betas 0.9 / 0.999, eps 1e-8) with lr_rot / lr_trans is applied. */
int mf_pose_refine_update(float* state, const float* c2w, const float* d_c2w, const float* losses, const float* loss_w,
                          double lr_rot, double lr_trans, int wait_iters, float* best_c2w, void* stream);
/* RO -> GO hand-off of tracking (mipsfusion.py:483-485,501-503), one 32-thread block: rot_cur (3,3) and trans_cur (3), the
 * RandomOptimizer's state, give c2w_out (4,4) = pose_compose(rot_cur, trans_cur) and go_state (32 floats, the layout above):
 * [0:4] matrix_to_quaternion(rot_cur) (standardised to a non-negative real part), [4:7] trans_cur, Adam moments and step
 * count 0, [22] = -1 (no best loss yet), [23] = [24] = 0 -- what FusedPoseRefiner.refine sets up on the host. */
int mf_track_handoff(const float* rot_cur, const float* trans_cur, float* c2w_out, float* go_state, void* stream);

/* ---- keyframe pose optimisation of the mapping loop (local_BA, mipsfusion.py:259-370: get_pose_param_optim :235-241,280-282,
 * pose_optimizer.step() every pose_accum_step iterations :338-342) on the device, one thread per pose.  state (K x 24 floats):
 * per pose [0:4] quaternion (w,x,y,z), [4:7] translation, [7:14] Adam m, [14:21] Adam v, [21] step count, [22:24] spare.
 * frozen (K uint8, NULL = none frozen): poses that are not parameters (the submap's first keyframe; the current frame unless
 * optim_cur); their poses_out entries are the input bit for bit and their state stays zero.
 * mf_ba_pose_init: poses (K,4,4) -> quaternion (pytorch3d matrix_to_quaternion, standardised to a non-negative real part) and
 * translation, zeroed moments and step; poses_out (K,4,4) = qt_to_transform_matrix of the parameters (geometry_helper.py:11-17). */
int mf_ba_pose_init(const float* poses, const uint8_t* frozen, int K, float* state, float* poses_out, void* stream);
/* One pose step: d_poses (K,4,4, rows 0-2 as mf_gen_rays_packed_bwd accumulates them) is pulled back to quaternion and
 * translation, one torch.optim.Adam step (betas 0.9 / 0.999, eps 1e-8, lr_rot / lr_trans) is applied, poses_out is rebuilt and
 * d_poses is zeroed (pose_optimizer.zero_grad()), frozen poses included. */
int mf_ba_pose_update(float* state, float* d_poses, const uint8_t* frozen, int K, double lr_rot, double lr_trans,
                      float* poses_out, void* stream);

/* ---- a13: RandomOptimizer particle scoring (RandomOptimizer.py:54-73,81-85,113-131) ----
 * particles6 (C_total,6) pre-sampled template; search_size (6), rot_cur (3,3), trans_cur (3) device;
 * dirs_cam (P,3) and target_d (P) are the sampled pixels.  c_begin/c_count select this rank's candidate
 * shard.  -> fitness (c_count), mean_sdf (c_count), pst7 (c_count,7) rescaled 7-D particles.
 * scratch: c_count*(P+12) floats. */
int mf_ro_score(const float* particles6, const float* search_size, const float* rot_cur, const float* trans_cur,
                const float* dirs_cam, const float* target_d, const mf_field* field_host, double trunc,
                double sdf_weight, int c_begin, int c_count, int P, float* fitness, float* mean_sdf, float* pst7,
                float* scratch, void* stream);
/* Steps 3-5 of RandomOptimizer.optimize (RandomOptimizer.py:202-224) on device, over all C candidates:
 * better mask, fitness-weighted mean transform, pose update, search-size update (in place).
 * better_mask (C) uint8; info (4) int32 = count_nonzero(better), success_flag, argmin(fitness), 0. */
int mf_ro_update(const float* fitness, const float* mean_sdf, const float* pst7, int C, double rescale,
                 float* rot_cur, float* trans_cur, float* search_size, uint8_t* better_mask, int32_t* info,
                 void* stream);
/* The same update reading the result of an all-gather in place: `gathered` = per-rank blocks of 9 * per floats
 * [fitness (per) | mean_sdf (per) | pst7 (per x 7)], candidate c in block c / per at row c % per (multi-GPU RandomOptimizer:
 * every rank's mf_ro_score writes one such block, one all-gather, no pack / unpack copies). */
int mf_ro_update_gathered(const float* gathered, int C, int per, double rescale, float* rot_cur, float* trans_cur,
                          float* search_size, uint8_t* better_mask, int32_t* info, void* stream);
/* Exchange + update in ONE kernel over NVLink peer memory (no collective call): peer_bases[r] = rank r's mapping of a
 * symmetric float arena holding, at float offset off_gathered, 2 x world x 9 x per floats (double-buffered gathered blocks) and,
 * at off_flags, `world` 32-bit sequence flags (zero-initialised).  The kernel stores `local_block` (this rank's 9 x per floats)
 * into every rank's gathered buffer, publishes `seq` (1, 2, 3, ... in lockstep on all ranks) in every rank's flags, waits for
 * all ranks' blocks and runs mf_ro_update on them.  A peer that never arrives sets the error flag (mf_tc_check_error). */
int mf_ro_update_peer(const float* local_block, const uint64_t* peer_bases, int world, int rank, int64_t off_gathered,
                      int64_t off_flags, unsigned int seq, int C, int per, double rescale, float* rot_cur, float* trans_cur,
                      float* search_size, uint8_t* better_mask, int32_t* info, void* stream);

/* ---- a14: joint multi-submap query + blend (model/Mesher.py:464-528,606-663; vis/math_helper.py:58-96) ----
 * Query points are either explicit (pts (G,3) fp64 world coordinates, as trimesh vertices) or a regular
 * grid given by its per-axis coordinates (the np.linspace arrays of Mesher.get_grid_uniform, Mesher.py:43-55),
 * generated on the fly with index = (iy*nx + ix)*nz + iz.  All pointers are device pointers.
 * g_begin/g_count select a contiguous range of the point index space (slab sharding across GPUs);
 * per-point outputs are indexed relative to g_begin. */
typedef struct {
    const double* pts;        /* NULL => regular grid */
    const double* ax; const double* ay; const double* az;
    int32_t nx, ny, nz;
} mf_point_set;

typedef struct {
    mf_field field;
    float w2l[12];            /* inverse(first_kf_pose)[:3,:4] row-major: world -> submap frame (geometry_helper.py:93-99) */
    double aabb_min[3], aabb_max[3];   /* inclusive containment test on fp64 coordinates (Mesher.py:168-175) */
    float centroid[3];
} mf_submap;

int64_t mf_joint_query_scratch_size(int64_t g_count);   /* bytes */
/* Pass 1: max_dist[m] = max over contained points of |x - centroid_m| (fp32; atomic max, so shards
 * can be combined with a max-reduction).  max_dist (M) must be zero-initialised by the caller. */
int mf_joint_query_maxdist(const mf_point_set* ps_host, const mf_submap* submaps_host, int M, int64_t g_begin,
                           int64_t g_count, float* max_dist, void* stream);
/* Pass 2, for submaps [m_begin, m_begin+m_count): acc (g_count,K) += w * value and w, K = 2 (sdf) or 4 (rgb);
 * w = exp(-10 clip(entropy,0,1e4)) * N(dist; 0, max_dist/3) for points inside the AABB (and vis != 0);
 * mask_any (g_count) |= contained & visible; contain (g_count,M) uint8 optional; vis (g_count,M) uint8 optional. */
int mf_joint_query_accumulate(const mf_point_set* ps_host, const mf_submap* submaps_host, int M, int m_begin,
                              int m_count, const float* max_dist, const uint8_t* vis, int color, int64_t g_begin,
                              int64_t g_count, float* acc, uint8_t* mask_any, uint8_t* contain, void* scratch,
                              void* stream);
/* Pass 3: out (g_count, K-1) = acc[:, :K-1] / acc[:, K-1] where mask_any (0 if the weight sum is 0), else the
 * fill value (-1 for sdf, 0 for rgb)  (Mesher.py:461,525-527). */
int mf_joint_query_finalize(const float* acc, const uint8_t* mask_any, int color, int64_t g_count, float* out, void* stream);

/* ---- N2: marching cubes on a dense SDF volume (external/NumpyMarchingCubes/marching_cubes/src/marching_cubes.cpp:418-462 =
 * marching_cubes(volume, isovalue, truncation) of utils/utils.py:78,159; binding replaced: pywrapper.cpp:9-54) ----
 * volume (nx,ny,nz) float32, C-contiguous, device (the reference reads each element as double and narrows it to float,
 * marching_cubes.cpp:82; the host side does that cast).  Results are bit-identical to the reference: vertices in voxel units in
 * the reference's order (first-come clusters on its 1e-5 lattice), faces in the i,j,k scan order with degenerate and duplicate
 * faces removed.  Two calls because the output sizes are data dependent:
 *   mf_mcubes_count : dual-node values, triangle count per cell and their scan offsets into `workspace`
 *                     (mf_mcubes_count_workspace_size bytes); *n_tris (device) = triangles before merging.  Asynchronous.
 *   mf_mcubes_mesh  : n_tris as read back by the caller; mesh_workspace of mf_mcubes_mesh_workspace_size(n_tris) bytes;
 *                     verts capacity (3 n_tris, 3) float32, faces capacity (n_tris, 3) uint32; counts (device, 3 x int64) =
 *                     {vertices, faces, clustering rounds}.  Synchronises `stream` once per clustering round (>= 1) and on return.
 * truncation must be finite; dimensions < 2048. */
int64_t mf_mcubes_count_workspace_size(int64_t nx, int64_t ny, int64_t nz);
int mf_mcubes_count(const float* volume, int64_t nx, int64_t ny, int64_t nz, float isovalue, float truncation, void* workspace,
                    int64_t* n_tris, void* stream);
int64_t mf_mcubes_mesh_workspace_size(int64_t n_tris);
int mf_mcubes_mesh(const void* count_workspace, int64_t nx, int64_t ny, int64_t nz, float isovalue, int64_t n_tris,
                   void* mesh_workspace, float* verts, uint32_t* faces, int64_t* counts, void* stream);

/* ---- N2 (cont.): mesh visibility filter of the Mesher (model/Mesher.py:247-281 point_mask, :221-231 get_face_mask;
 * helper_functions/geometry_helper.py:216-222 project_to_pixel) ----
 * points (n,3) world; w2c (k,12): rows of the inverse keyframe poses [R | t]; max_depth (k): largest stored depth of each
 * keyframe (Mesher.py:273); K (9) camera matrix, all fp32 device.  seen[i] = 1 iff for some keyframe the point projects
 * strictly inside (edge, img_w - edge) x (edge, img_h - edge), has camera z < 0 and 0 < |z| < max_depth; fp32 in the
 * reference's operation order (left-to-right sums of products, x negated before K, division by z + 1e-5).
 * mf_mesh_face_mask: keep[f] = seen[a] | seen[b] | seen[c] (a face is dropped only if all three vertices are unseen). */
int mf_mesh_seen_mask(const float* points, int64_t n, const float* w2c, const float* max_depth, int k, const float* K, int img_w,
                      int img_h, int edge, uint8_t* seen, void* stream);
int mf_mesh_face_mask(const uint8_t* seen, const int64_t* faces, int64_t n_faces, uint8_t* keep, void* stream);

/* ---- a15: overlap-region SDF consistency of the inactive-map global BA (InactiveMap.py:128-139 infer_pts, :149-165
 * get_SDF_dif, :177-192 get_SDF_dif2; loss helper_functions/geometry_helper.py:225-229), P submap pairs x N rays ----
 * pair_tab (P,4) int32 device: {pose1, pose2, off1, off2} = rows of the two first-keyframe poses in first_poses (K,4,4) and
 * the first row of each side's N points in pts / raw / d_raw / d_pts (2 P N rows in all, grouped by submap by the caller).
 * Element (p, r) of target_d is target_d[(p N + r) ld_d], its direction rays_d_cam[(p N + r) ld_dir + 0..2].  ovlp: the
 * overlap keyframe poses, (P, N, 4, 4) when ovlp_per_ray, else (P, 1, 4, 4).  All fp32 device, no atomics (deterministic).
 * mf_overlap_points: finv (P,2,16) = first_poses[pose_s]^-1 (fp64 adjugate / determinant, rounded once to fp32);
 *   A = finv O (fp32), pts[off_s + r] = A[:3,3] + (sum_k d_cam[k] A[:3,k]) depth (InactiveMap.py:128-139). */
int mf_overlap_points(const float* first_poses, const int* pair_tab, int P, int N, const float* ovlp, int ovlp_per_ray,
                      const float* target_d, int ld_d, const float* rays_d_cam, int ld_dir, float* finv, float* pts, void* stream);
/* mf_overlap_loss: raw = the field outputs of pts (mf_field_query, per submap segment); sdf = raw[:,3] trunc;
 * loss[p] = sum_r (sdf1 m - sdf2 m)^2 / (count_nonzero(m) + 0.001) (geometry_helper.py:225-229), fixed-order reduction.
 * mask_kind 0: m = (target_d > 0) (get_SDF_dif, InactiveMap.py:149-165); 1: float mask[(p N + r) ld_m]; 2: uint8/bool mask
 * (get_SDF_dif2, :177-192).  d_raw (2 P N, 10): d loss[p] / d raw for an upstream gradient of 1, only column 3 non-zero,
 * rows with m = 0 exactly zero (the field backward skips them). */
int mf_overlap_loss(const float* raw, const int* pair_tab, int P, int N, const float* target_d, int ld_d, const void* mask,
                    int mask_kind, int ld_m, double trunc, float* loss, float* d_raw, void* stream);
/* mf_overlap_pose_bwd: d_pts = mf_field_query_bwd of d_raw (point gradients only); g_loss[p ld_g] the upstream gradient of
 * loss[p] (ld_g = 0: one shared value; NULL = 1).  dA = d loss / d A (dA[:3,3] = dx, dA[i][k] = dx_i depth d_cam_k); dF_pair (P,2,16) scratch receives
 * -finv^T (sum_r dA_r O_r^T) finv^T; d_first (n_poses,4,4) = sum over pairs in pair order (side 1, then side 2) of the sides
 * that use each pose (written, not accumulated); d_ovlp (same shape as ovlp, optional) = sum_s finv_s^T dA_s. */
int mf_overlap_pose_bwd(const float* finv, const int* pair_tab, int P, int N, const float* ovlp, int ovlp_per_ray,
                        const float* target_d, int ld_d, const float* rays_d_cam, int ld_dir, const float* d_pts,
                        const float* g_loss, int ld_g, int n_poses, float* dF_pair, float* d_first, float* d_ovlp, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MIPSFUSION_B200_H */
