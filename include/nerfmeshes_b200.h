/*
 * nerfmeshes_b200 — C ABI of the B200-native NeRF render / dense-grid hot path.
 *
 * The reference (qway/nerfmeshes, pure Python) has no FFI layer; its de-facto operator API for this path
 * is the Python surface SURVEY.md section 8(b) lists.  Each entry point below names the reference interface it
 * replaces (paths relative to /root/reference/).  The reference-side binding a maintainer would add is a
 * ctypes stub; it is shown in INTEGRATION.md and shipped as nerfmeshes_b200/_lib.py.
 *
 * Conventions
 *   - plain C: pointers + sizes, no torch / C++ types.  `stream` is a cudaStream_t passed as void* (NULL =
 *     legacy default stream).
 *   - every call returns 0 on success, <0 on error; nm_last_error() returns a thread-local message.
 *   - pointers suffixed _dev are device pointers on the handle's device, _host are host pointers.
 *   - device-pointer calls are stream-ordered and asynchronous w.r.t. the host; *_host calls synchronise
 *     before returning (they copy results back).
 *   - the handle owns packed weights, tables, the voxel list and a grow-only workspace; callers own all
 *     input / output buffers.  One host thread per handle at a time.
 */
#ifndef NERFMESHES_B200_H
#define NERFMESHES_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NM_VERSION 100 /* 0.1.0 */

/* Shape of one FlexibleNeRFModel — constructor arguments of src/nerf/models.py:5-22. */
typedef struct NmNetDesc {
  int32_t num_layers;          /* 8  */
  int32_t hidden_size;         /* 256 (128 or 256 supported by the tensor-core path) */
  int32_t skip_step;           /* 4  */
  int32_t num_encoding_fn_xyz; /* 10 */
  int32_t num_encoding_fn_dir; /* 4  */
  int32_t include_input_xyz;   /* 1  */
  int32_t include_input_dir;   /* 1  */
  int32_t log_sampling_xyz;    /* 1  */
  int32_t log_sampling_dir;    /* 1  */
  int32_t use_viewdirs;        /* 1  */
} NmNetDesc;

/* MLP arithmetic selection (SURVEY 7.3.1). */
enum {
  NM_PREC_EXACT = 0, /* tcgen05, fp16 hi/lo split operands, 3 MMAs per product, fp32 accumulate (default) */
  NM_PREC_FAST = 1,  /* tcgen05, single fp16 operands (misses the 1e-4 target; for comparison only)      */
  NM_PREC_FP32 = 2   /* CUDA-core fp32 FMA kernel (bit-for-bit fp32 arithmetic; slow; debugging yard-stick) */
};

/* cfg.nerf.{train,validation}.* and cfg.dataset.* knobs read on the path (config/nerf-synthetic-lego.yml). */
typedef struct NmRenderCfg {
  int32_t num_coarse;          /* cfg.nerf.train.num_coarse (the reference sizes its samplers from .train,
                                  src/models/model_nerf.py:31-32)                                        */
  int32_t num_fine;            /* cfg.nerf.train.num_fine; 0 = coarse only (models.use_fine False)          */
  int32_t lindisp;
  int32_t perturb;             /* stratified jitter / random u (distributional parity only)                 */
  int32_t white_background;
  float noise_std;             /* radiance_field_noise_std of the active mode                              */
  float attenuation_threshold; /* 1e-5, src/models/model_base.py:28-33                                     */
  int32_t precision;           /* NM_PREC_*                                                                */
  int32_t act_scale_log2;      /* s >= 0: fp16 A-operands are stored as x * 2^-s (range guard, SURVEY 7.3.1)  */
} NmRenderCfg;

typedef struct NmHandle_t* NmHandle;

enum { NM_NET_COARSE = 0, NM_NET_FINE = 1 };

/* Output block of one render call: the fields of OutputBundle (src/nerf/modules.py:40-47).  Any pointer may be
 * NULL (that output is skipped).  depth is the eval-mode thresholded map (modules.py:108-109) unless flag
 * NM_FLAG_TRAINING is set; depth_raw is sum(w*t) before the threshold (what parity tests compare). */
typedef struct NmRenderOut {
  float* rgb;          /* (R,3) */
  float* depth;        /* (R,)  */
  float* depth_raw;    /* (R,)  */
  float* acc;          /* (R,)  */
  float* disp;         /* (R,)  */
  float* weights;      /* (R,S) S = num_coarse+num_fine (or num_coarse when coarse-only / BuFF) */
  float* mask_weights; /* (R,S) */
  float* t_vals;       /* (R,S) the sample distances actually used (debug / parity) */
  float* coarse_rgb;   /* (R,3) coarse-pass colour (training loss needs it, model_nerf.py:128) */
  float* coarse_acc;   /* (R,)  */
  float* coarse_disp;  /* (R,)  */
  float* coarse_weights; /* (R,num_coarse) */
} NmRenderOut;

enum {
  NM_FLAG_TRAINING = 1,    /* module.training: no depth threshold, train noise_std            */
  NM_FLAG_BUFF = 2,        /* BuFFModel.forward: AABB-clipped sampling, single net (coarse slot) */
  NM_FLAG_TEACHER_T = 4,   /* t_vals is an INPUT: skip sampling, run net `which`=fine-if-present on it */
  NM_FLAG_RANDOM_VOXELS = 8 /* with NM_FLAG_BUFF: cfg.tree.use_random_sampling — multinomial voxel draws + uniform depth inside
                               the voxel (src/nerf/tree.py:280-297) instead of the deterministic placement; uses `seed` */
};

/* ---- lifecycle -------------------------------------------------------------------------------------- */
int nm_version(void);
const char* nm_last_error(void);
/* 0 if `device` is a compute-capability-10.x GPU, error otherwise (the library fails loudly elsewhere). */
int nm_device_check(int device);
/* Replaces NeRFModel.__init__/BuFFModel.__init__ (src/models/model_nerf.py:24-32, model_buff.py:13-29). */
int nm_create(int device, const NmNetDesc* coarse, const NmNetDesc* fine_or_null, const NmRenderCfg* cfg,
              NmHandle* out);
int nm_destroy(NmHandle h);
int nm_set_render_cfg(NmHandle h, const NmRenderCfg* cfg);

/* Replaces load_state_dict for one FlexibleNeRFModel (weight ABI: SURVEY Appendix A.1).  names[i] is the
 * reference state-dict key without the model prefix ("layer1.weight", "layers_xyz.4.bias", "fc_alpha.weight",
 * ...); tensors_host[i] points at numel[i] fp32 values in the reference (out,in) row-major layout. */
int nm_load_weights(NmHandle h, int which, int n_tensors, const char* const* names,
                    const float* const* tensors_host, const int64_t* numel);
/* Same, with the tensors already in device memory (fp32, contiguous): transposes / packs on the device, stream-ordered,
 * no host round trip — the per-step weight refresh of a training loop whose optimiser updates CUDA parameters. */
int nm_load_weights_dev(NmHandle h, int which, int n_tensors, const char* const* names,
                        const float* const* tensors_dev, const int64_t* numel, void* stream);
/* Sampler tables: coarse s = torch.linspace(0,1,num_coarse) (src/nerf/modules.py:154) and the SamplePDF buffer
 * u = torch.linspace(0,1,num_fine) (modules.py:193).  Host pointers; NULL = recompute i/(n-1) in fp32. */
int nm_set_tables(NmHandle h, const float* coarse_s_host, const float* fine_u_host);
/* BuFF voxel list, checkpoint['tree']['voxels'] (V,2,3) (src/nerf/tree.py:345-358). */
int nm_set_tree(NmHandle h, const float* voxels_host, int32_t V);

/* ---- hot path, device pointers ---------------------------------------------------------------------- */
/* BaseModel.sample_points (src/models/model_base.py:65-73) == FlexibleNeRFModel.forward (src/nerf/models.py:60-80).
 * pts/dirs (M,3) fp32; out (M,4) = [sigmoid rgb, raw sigma], or (M,) raw sigma when sigma_only. */
int nm_point_mlp(NmHandle h, int which, const float* pts_dev, const float* dirs_dev, int64_t M, float* out_dev,
                 int sigma_only, void* stream);
/* NeRFModel.forward / BuFFModel.forward (src/models/model_nerf.py:37-78, model_buff.py:34-69).
 * origins: o_stride = 0 -> one shared (3,) origin, 3 -> per-ray (R,3).  near/far: nf_stride = 0 -> 2 scalars in
 * near_far_host[0..1]; 1 -> per-ray near (R,) and far (R,) device arrays in near_dev / far_dev. */
int nm_render_rays(NmHandle h, const float* origins_dev, int o_stride, const float* dirs_dev, int64_t R,
                   const float* near_far_host, const float* near_dev, const float* far_dev, int flags, uint64_t seed,
                   const NmRenderOut* out_dev, void* stream);
/* get_ray_bundle (+ ndc_rays) fused with the render for image rows [row0,row1) — the eval_nerf.py:50-98 image
 * loop with the pose, not 7.7 MB of directions, crossing PCIe.  pose_host: 12 floats, c2w[:3,:4] row-major.
 * Outputs are (row1-row0)*W rays. */
int nm_render_image(NmHandle h, const float* pose_host, int H, int W, float focal, int ndc, int row0, int row1,
                    const float* near_far_host, int flags, uint64_t seed, const NmRenderOut* out_dev, void* stream);
/* get_ray_bundle / ndc_rays alone (src/nerf/nerf_helpers.py:226-307): dirs (rows,W,3); origins (rows,W,3) only
 * when ndc (else the origin is pose[:,3]). */
int nm_ray_bundle(NmHandle h, const float* pose_host, int H, int W, float focal, int ndc, float ndc_near, int row0,
                  int row1, float* origins_dev_or_null, float* dirs_dev, void* stream);
/* ndc_rays(H, W, focal, near, rays_o, rays_d) on caller-supplied rays (src/nerf/nerf_helpers.py:280-307, called positionally
 * by DataBundle.ndc, src/data/data_helpers.py:164-167): n rays, origins with o_stride 0 (one shared origin) or 3. */
int nm_ndc_rays(NmHandle h, int H, int W, float focal, float near, const float* origins_dev, int o_stride,
                const float* dirs_dev, int64_t n, float* origins_out_dev, float* dirs_out_dev, void* stream);
/* extract_radiance (src/mesh_nerf.py:27-53) for grid planes [x0,x1): points from the three linspace tables
 * (host, lengths n0,n1,n2; pass torch.linspace values for bit-identical coordinates), dirs := positions.
 * sigma_dev (x1-x0,n1,n2) raw density; rgb_dev (x1-x0,n1,n2,3) or NULL (sigma-only fast path). */
int nm_grid_sigma(NmHandle h, const float* lin0_host, const float* lin1_host, const float* lin2_host, int n0, int n1,
                  int n2, int x0, int x1, float* sigma_dev, float* rgb_dev_or_null, void* stream);
/* numpy min / max / std of a float32 volume (extract_iso_level, src/mesh_nerf.py:56-65): out_host[0..2] =
 * {min, max, std}; synchronises. */
int nm_volume_stats(NmHandle h, const float* vol_dev, int64_t n, float* out_host);

/* The same statistics for a volume sharded over several GPUs, stream-ordered and without host synchronisation: pass 1 writes
 * out_dev[0..2] = {min, max, sum} of this shard (doubles), pass 2 writes out_dev[3] = sum (x - *mean_dev)^2; the caller
 * combines the shards between and after the passes (all_gather / all_reduce on the device values). */
int nm_volume_stats_dev(NmHandle h, const float* vol_dev, int64_t n, int pass, const double* mean_dev, double* out_dev, void* stream);

/* skimage.measure.marching_cubes(volume, level) seam (src/mesh_nerf.py:79) on a device volume (nx,ny,nz) fp32, Lewiner-style
 * topology resolution (face / interior tests, cell-centre vertices): sign bit-volume -> count -> scan -> emit.  Two-call
 * protocol: nm_marching_cubes_count fills counts_host = {n_vertices, n_triangles} (synchronises);
 * nm_marching_cubes_emit (same volume and iso) writes verts (n_vertices,3) fp32 in index coordinates (x_off, an integer,
 * added to axis 0), normals (n_vertices,3), faces (n_triangles,3) int32.  Indexed mesh: one vertex per crossed grid edge
 * plus the centre vertices, ordered by owning grid point. */
int nm_marching_cubes_count(NmHandle h, const float* vol_dev, int nx, int ny, int nz, float iso,
                            int64_t* counts_host, void* stream);
int nm_marching_cubes_emit(NmHandle h, const float* vol_dev, int nx, int ny, int nz, float iso, float x_off,
                           float* verts_dev, float* normals_dev, int32_t* faces_dev, void* stream);
/* The same for ONE SHARD of a grid split along axis 0 (mesh_nerf.py:27-92 on N GPUs, SURVEY 8e): the buffer holds global
 * planes [g_x0, g_x0+nb) of a grid with g_nx planes and the call owns the grid points of buffer planes [p_lo,p_hi): it
 * emits their vertices and the triangles of their cells.  The buffer must also hold, where they exist globally, plane
 * p_hi (cells of the last owned layer), p_hi+1 and p_lo-1 (gradient normals): halo planes, received from the neighbours or
 * recomputed.  Face indices are v_base + local id, and ids of plane-p_hi vertices (owned by the next shard) continue the
 * local numbering; with v_base = the exclusive scan of the shards' n_vertices, the concatenated shard outputs ARE the
 * single-GPU arrays, bit for bit (no duplicate vertices, nothing to de-duplicate). */
int nm_mc_count(NmHandle h, const float* vol_dev, int nb, int ny, int nz, float iso, int g_x0, int g_nx, int p_lo, int p_hi,
                int64_t* counts_host, void* stream);
int nm_mc_emit(NmHandle h, const float* vol_dev, int nb, int ny, int nz, float iso, int g_x0, int g_nx, int p_lo, int p_hi,
               int64_t v_base, float* verts_dev, float* normals_dev, int32_t* faces_dev, void* stream);

/* Replaces export_obj (src/nerf/nerf_helpers.py:86-111): `v x y z [r g b]`, `vn x y z`, `f i//i j//j k//k` (1-based) with
 * byte-identical number formatting (python repr of the float32 widened to double).  Host arrays, no GPU involved;
 * diffuse may be NULL or shorter than the vertex list (vertices beyond it get no colour, like the reference's
 * len(diffuse) > idx test). */
int nm_export_obj(const char* path, const float* verts_host, int64_t n_verts, const int32_t* faces_host, int64_t n_faces,
                  const float* diffuse_host, int64_t n_diffuse, const float* normals_host, int64_t n_normals);

/* ---- mesh-quality metrics (the Chamfer metric of BaseModel.validation_epoch_end, src/models/model_base.py:82-102) ----- */
/* The nearest-neighbour step of pytorch3d.loss.chamfer_distance (model_base.py:99): for each x_i of x (N,3) fp32, dist (N,)
 * = min_j |x_i - y_j|^2 over y (M,3) fp32 and idx (N,) int32 = the argmin.  One pair's distance is
 * ((dx*dx) + (dy*dy)) + (dz*dz), d = x - y, every operation rounded to nearest in fp32, no FMA contraction (a float32 numpy
 * brute force reproduces it bit for bit); a tie goes to the lowest j, independent of how the work is split.  M >= 1,
 * M < 2^31.  Exact brute force, N*M pair evaluations. */
int nm_nearest(NmHandle h, const float* x_dev, int64_t N, const float* y_dev, int64_t M, float* dist_dev, int32_t* idx_dev,
               void* stream);
/* pytorch3d.ops.sample_points_from_meshes for one mesh (model_base.py:95-97): n points drawn on the surface of verts (V,3)
 * fp32 / faces (F,3) int32 (indices in [0,V), not checked on the device), a face with probability proportional to its area
 * 1/2|(v1-v0)x(v2-v0)| (with replacement), then p = w0 v0 + w1 v1 + w2 v2 with w0 = 1-sqrt(u), w1 = sqrt(u)(1-v),
 * w2 = sqrt(u) v.  points (n,3); face_idx (n,) int32 and normals (n,3) (the sampled face's unit normal) may be NULL.  A mesh
 * without faces or without area gives zero points and normals and face index -1.  Counter-based draws from `seed`: the
 * same seed gives the same samples.  The area CDF (fp64, 8 bytes per face) lives in the handle's workspace. */
int nm_mesh_sample(NmHandle h, const float* verts_dev, int64_t V, const int32_t* faces_dev, int64_t F, int64_t n, uint64_t seed,
                   float* points_dev, int32_t* face_idx_dev_or_null, float* normals_dev_or_null, void* stream);

/* ---- hot path, host buffers (what a reference-side caller holding CPU tensors binds) ------------------ */
/* model.query(ray_batch) with host tensors (src/eval_nerf.py:62-69): copies H2D, renders, copies D2H, syncs. */
int nm_query_host(NmHandle h, const float* origins_host, int o_stride, const float* dirs_host, int64_t R,
                  const float* near_far_host, int flags, uint64_t seed, const NmRenderOut* out_host);
/* one image from a pose, results to host (eval_nerf.py image loop). */
int nm_render_image_host(NmHandle h, const float* pose_host, int H, int W, float focal, int ndc, int row0, int row1,
                         const float* near_far_host, int flags, uint64_t seed, const NmRenderOut* out_host);
/* model.sample_points with host tensors (src/mesh_nerf.py:43-48). */
int nm_point_mlp_host(NmHandle h, int which, const float* pts_host, const float* dirs_host, int64_t M,
                      float* out_host, int sigma_only);

/* ---- training (SURVEY §8f-1) --------------------------------------------------------------------------
 * Replaces `loss.backward()` of NeRFModel.training_step / BuFFModel.training_step (src/models/model_nerf.py:88-151,
 * model_buff.py) for the parameters of both FlexibleNeRFModels: gradients flow from the bundles' rgb_map through
 * VolumeRenderer (src/nerf/modules.py:67-121) and the network (src/nerf/models.py:60-80); SamplePDF is detached
 * (modules.py:201).  The call re-runs the forward for these rays (same flags + seed => same samples and noise) and
 * ACCUMULATES dL/dtheta into the handle's gradient buffers (fp32, atomics: summation order is not reproducible).
 *   nm_backward_rays : d_rgb_dev (R,3) = dL/d rgb_map of the main bundle (fine, or the only one);
 *                      d_coarse_rgb_dev (R,3) or NULL = dL/d coarse rgb_map (two-network NeRF only).
 *   nm_loss_backward : the reference's loss itself, mse(coarse.rgb_map, target) + mse(fine.rgb_map, target)
 *                      (mean over R*3); loss_dev (2 floats, device, or NULL) += {coarse-or-only term, fine term}.
 *   nm_get_grad      : copies the gradient of one state-dict tensor (SURVEY A.1 names, reference (out,in) layout)
 *                      into out_dev.
 * Loss terms other than rgb_map (depth, acc, weights) carry no gradient here; the reference has none. */
int nm_zero_grad(NmHandle h, void* stream);
int nm_backward_rays(NmHandle h, const float* origins_dev, int o_stride, const float* dirs_dev, int64_t R,
                     const float* near_far_host, const float* near_dev, const float* far_dev, int flags, uint64_t seed,
                     const float* d_rgb_dev, const float* d_coarse_rgb_dev, void* stream);
int nm_loss_backward(NmHandle h, const float* origins_dev, int o_stride, const float* dirs_dev, int64_t R,
                     const float* near_far_host, const float* near_dev, const float* far_dev, int flags, uint64_t seed,
                     const float* target_rgb_dev, float* loss_dev, void* stream);
int nm_get_grad(NmHandle h, int which, const char* name, float* out_dev, int64_t numel, void* stream);

/* ---- BuFF tree maintenance (SURVEY §8f rank 4) ----------------------------------------------------------
 * nm_ray_voxel_indices: the `indices` output of TreeSampling.batch_ray_voxel_intersect (src/nerf/tree.py:215-343,
 *   deterministic branch) for cfg.num_coarse samples per ray: the voxel (row of the nm_set_tree list) every sample lies
 *   in, int32 (R,S), -1 on rays that hit no voxel; z_out_dev (R,S) optionally receives the sample distances with the
 *   uniform fallback on those rays (model_buff.py:52-53).  _ex: flags = NM_FLAG_RANDOM_VOXELS selects the random branch
 *   (tree.py:280-297) with `seed` — pass the seed of the render call whose samples are being attributed.
 * nm_tree_integrate: TreeSampling.ray_batch_integration (tree.py:177-206) past its step gate: memm[v] +=
 *   (sum of weights / sum of weight masks of the samples in v - memm[v]) / counter for every voxel that received a sample.
 *   idx/weights/mask: n = R*S entries (whole batch, idx -1 skipped, or only the rows of rays that hit). */
int nm_ray_voxel_indices(NmHandle h, const float* origins_dev, int o_stride, const float* dirs_dev, int64_t R,
                         const float* near_far_host, float* z_out_dev, int32_t* idx_out_dev, void* stream);
int nm_ray_voxel_indices_ex(NmHandle h, const float* origins_dev, int o_stride, const float* dirs_dev, int64_t R,
                            const float* near_far_host, int flags, uint64_t seed, float* z_out_dev, int32_t* idx_out_dev,
                            void* stream);
int nm_tree_integrate(NmHandle h, const int32_t* idx_dev, const float* weights_dev, const float* mask_weights_dev, int64_t n,
                      float* memm_dev, int32_t V, int32_t counter, void* stream);

/* Test hook for the tensor-core GEMM of the backward pass (nm_gemm_tc.cu): D (M,N) = A (M,K) B (N,K)^T from fp32
 * row-major device arrays through the bf16 hi/lo operand packs.  a_cols / b_cols: that operand is given transposed
 * ((K,M) / (K,N)) and packed along its rows (the weight-gradient operands; 1 = K-major tiles, 2 = MN-major tiles read
 * through MN-major shared-memory descriptors); k_split: feed K as two segments;
 * fp16: fp16 halves instead of bf16; atomic: D += with K split over CTAs. */
int nm_debug_gemm(NmHandle h, const float* a_dev, const float* b_dev, int M, int N, int K, int a_cols, int b_cols,
                  int k_split, int n_passes, int fp16, int atomic, float* d_dev, void* stream);

/* ---- host-only debugging aid (no CUDA): the layer program + tensor-core weight stream nm_load_weights would
 * upload, for CPU tests of the schedule / swizzle logic.  program_out receives the internal NetProgram struct
 * (nerfmeshes_b200/csrc/nm_program.h). */
int nm_debug_pack(const NmNetDesc* desc, int n_tensors, const char* const* names, const float* const* tensors_host,
                  const int64_t* numel, int sigma_only, void* program_out, size_t program_cap, uint8_t* pack_out,
                  size_t pack_cap, size_t* pack_need);

/* Host-only: how the fused compositor deals tiles to CTAs for `samples_per_ray` samples (nm_mlp_tc.cu).  Returns the group
 * size g = lcm(S,128)/128 (0: the fused compositor is not used for this S); if tiles_out != NULL it receives the tile
 * indices CTA `cta` of `grid` CTAs processes, in order, for a launch of n_tiles tiles (at most cap entries; *n_out = count). */
int nm_debug_tile_schedule(int samples_per_ray, int64_t n_tiles, int grid, int cta, int64_t* tiles_out, int64_t cap, int64_t* n_out);

/* Device-side error flags, readable even after a kernel trapped: out2[0] = tcgen05 pipeline watchdog code (0 = ok),
 * out2[1] = AABB hit-list overflow. */
int nm_kernel_flags(NmHandle h, int32_t* out2);
/* Synchronises `stream`, then fails (<0, message in nm_last_error) if a kernel of this handle raised a device-side flag.
 * The asynchronous device-pointer entry points report flags raised by EARLIER calls when they are entered; *_host calls
 * check before they return. */
int nm_check_flags(NmHandle h, void* stream);

/* ---- introspection ---------------------------------------------------------------------------------- */
/* number of kernels launched through this handle since creation (bench.py's gpu_launches). */
int64_t nm_launch_count(NmHandle h);
/* duration in ms of the last fused-MLP launch sequence, measured with CUDA events on the call's stream when
 * timing is enabled (bench.py's roofline); <0 if disabled. */
int nm_set_timing(NmHandle h, int enable);
double nm_mlp_time_ms(NmHandle h, int64_t* points_out, int64_t* launches_out);

#ifdef __cplusplus
}
#endif
#endif /* NERFMESHES_B200_H */
