/*
 * vggsfm_b200 -- C ABI of the B200-native geometry hot path for VGGSfM.
 *
 * The reference (facebookresearch/vggsfm @ e1d9d2e) has no FFI of its own: its seam for this path
 * is ordinary Python symbols plus the pycolmap object API (SURVEY.md section 8b).  Every entry
 * point below names the reference call site it replaces.  All pointers are DEVICE pointers owned
 * by the caller unless marked "host"; `stream` is a cudaStream_t passed as void*; no entry point
 * allocates device memory (the caller passes a workspace sized by the matching *_workspace_bytes).
 * Return value: 0 on success, negative VGG_E* on error; vgg_last_error() gives the message.
 *
 * Layouts (row-major, densely packed):
 *   observations  uv   float  [S,N,2]   pixels (or normalised coordinates where stated)
 *                 mask uint8  [S,N]     1 = observation participates
 *   cameras       poses  double [S,12]  cam_from_world R|t, 3x4 row-major
 *                 intr   double [S,4]   f, cx, cy, k   (k unused for SIMPLE_PINHOLE)
 *   points        double [N,3]
 */
#ifndef VGGSFM_B200_H
#define VGGSFM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VGG_OK 0
#define VGG_EINVAL (-1)
#define VGG_ECUDA (-2)
#define VGG_EWORKSPACE (-3)
#define VGG_ESOLVER (-4)

#define VGG_SIMPLE_PINHOLE 0
#define VGG_SIMPLE_RADIAL 1

#define VGG_INTR_CONST 0      /* intrinsics held constant (video_runner.py:813-815)            */
#define VGG_INTR_PER_FRAME 1  /* one pycolmap.Camera per frame (tensor_to_pycolmap.py:78-110)  */
#define VGG_INTR_SHARED 2     /* shared_camera=True: one Camera for all frames                 */

const char* vgg_last_error(void);
int vgg_version(void);

/* ------------------------------------------------------------------------------------------- */
/* Bundle adjustment: replaces pycolmap.bundle_adjustment(reconstruction, ba_options)           */
/* (vggsfm/utils/triangulation.py:213,1050,1142; vggsfm/runners/video_runner.py:508,1321-1331)  */
/* and the tensor<->Reconstruction marshalling around it (tensor_to_pycolmap.py:16-214).        */
/* ------------------------------------------------------------------------------------------- */

typedef struct vgg_ba_problem {
  int32_t S, N;
  int32_t camera_model;        /* VGG_SIMPLE_* */
  int32_t intr_mode;           /* VGG_INTR_*   */
  const float* uv;             /* [S,N,2] pixels */
  const uint8_t* mask;         /* [S,N] */
  const uint8_t* param_const;  /* [S*dc+ns] 1 = reduced parameter held constant (gauge, fixed poses) */
  const uint8_t* point_const;  /* [N] 1 = point held constant (video_runner.py:821-829), or NULL */
  double* poses;               /* [S,12] in/out */
  double* intr;                /* [S,4]  in/out */
  double* points;              /* [N,3]  in/out */
} vgg_ba_problem;

/* Ceres solver options as COLMAP's BundleAdjustmentOptions sets them (triangulation_helpers.py:626-635). */
typedef struct vgg_ba_options {
  int32_t max_num_iterations;
  int32_t max_num_consecutive_invalid_steps;
  int32_t jacobi_scaling;
  int32_t reserved;
  double function_tolerance, gradient_tolerance, parameter_tolerance;
  double initial_trust_region_radius, max_trust_region_radius, min_trust_region_radius;
  double min_relative_decrease, min_lm_diagonal, max_lm_diagonal;
} vgg_ba_options;

typedef struct vgg_ba_summary {
  int32_t iterations, successful, termination, reserved;
  double initial_cost, final_cost, final_radius;
  double device_ms;            /* CUDA-event time of the LM loop on `stream` */
  int64_t kernel_launches;     /* kernels of this library launched by the call */
} vgg_ba_summary;

/* termination codes */
#define VGG_BA_NO_CONVERGENCE 0
#define VGG_BA_CONVERGENCE_GRADIENT 1
#define VGG_BA_CONVERGENCE_FUNCTION 2
#define VGG_BA_CONVERGENCE_PARAMETER 3
#define VGG_BA_MIN_TRUST_REGION 4
#define VGG_BA_FAILURE 5

/* Sum/max all-reduce hook over track shards (one process per GPU).  `buf` is a device pointer
 * inside the caller's workspace; op 0 = sum, 1 = max, 2 = barrier across ranks on `stream` (buf NULL).
 * NULL = single GPU. */
typedef int (*vgg_allreduce_fn)(void* user, double* buf, size_t count, int op, void* stream);

/* Fused reduction over NVLink/NVSwitch: the reduced camera system lives in symmetric (peer-mapped) memory and
 * every rank's assemble / Schur kernels add their contributions with multimem.red on the multicast address,
 * so the per-iteration all-reduce of [D x Dpad | rhs | diag | g] needs no separate collective.  ar_local and
 * ar_multicast address the same allocation (e.g. torch.distributed._symmetric_memory). */
typedef struct vgg_ba_fabric {
  double* ar_local;
  double* ar_multicast;
  size_t ar_doubles;     /* >= vgg_ba_reduced_system_doubles() */
  /* v2 (optional; world = 0 keeps v1): reduce-scatter of the lower triangle's 128-row blocks onto their owners
   * (block b -> rank b mod world) with system-scope REDs over NVLink, gather by peer loads, barriers and the small
   * cost/gradient all-reduces as kernels on the same allocation -- no NCCL call, no host callback inside the LM loop,
   * inbound traffic per GPU independent of the number of ranks, bit-identical systems on all ranks.
   * peer_base[r] = rank r's base address of the SAME symmetric allocation (ar_local == peer_base[rank]), which must
   * hold total_doubles >= vgg_ba_fabric_doubles() and be zero-filled once when it is created. */
  int32_t world, rank;
  double* peer_base[8];
  size_t total_doubles;
} vgg_ba_fabric;

void vgg_ba_default_options(vgg_ba_options* opt);
int vgg_ba_dims(int camera_model, int intr_mode, int* dc, int* ns);
int vgg_ba_workspace_bytes(int S, int N, int camera_model, int intr_mode, size_t* bytes);

/* Fused residual + analytic 2x(dc+3) Jacobian + normal-equation block kernel (one launch).
 * Outputs (all double): cost[1]; camrec[S,KR] = per frame (g_c[dc] | H_cc upper-packed | H_cs[6,ns]);
 * g_p[N,3]; H_pp[N,6] (xx,xy,xz,yy,yz,zz); W[N, pitch, 3] track-major coupling blocks J_c^T J_p with
 * row = s*dc+i (shared-intrinsics rows at S*dc..) and pitch = D rounded up to even, D = S*dc+ns;
 * shared[8] = (g_s[2], H_ss xx,xy,yy).  KR = vgg_ba_camrec_len().  The last int argument is the number of
 * tracks each warp walks (0 = choose). */
int vgg_ba_camrec_len(int camera_model, int intr_mode);
int vgg_ba_build_blocks(const vgg_ba_problem* prob, double* cost, double* camrec, double* g_p,
                        double* H_pp, double* W, double* shared, int tracks_per_warp, void* stream);

/* Schur complement of the point blocks onto the camera system (second kernel of the path):
 * given the blocks above, the Jacobi scales and the trust-region radius, writes
 * Sraw[D,Dpad] (symmetric, both triangles written) = H_cc - sum_j W_j V_j^-1 W_j^T and rhs[Dpad] =
 * -(g_c - sum_j W_j V_j^-1 g_pj).  Exposed for the parity tests and profiling. */
int vgg_ba_schur(const vgg_ba_problem* prob, const double* camrec, const double* g_p,
                 const double* H_pp, const double* W, const double* shared, const double* scale_p,
                 double radius, double min_diag, double max_diag, void* workspace, size_t ws_bytes,
                 double* Sraw, double* rhs, int* Dpad_out, void* stream);

/* Blocked Cholesky of the reduced camera system (csrc/chol.cu): in-place factorisation of the row-major
 * lower triangle of A [n x n], leading dimension lda (even), replacing the potrf inside Ceres' DENSE_SCHUR.  On
 * return the lower triangle holds L and the strict upper triangle L^T.
 * workspace >= ceil(n/128)*131072 + 1024 bytes (n <= 24000); *info_host = 0, the 1-based index of the failing pivot, or
 * INT_MAX if the in-kernel hand-off between CTAs stalled (bounded spin; never seen, reported instead of hanging). */
int vgg_cholesky_lower(int n, int lda, double* A, void* workspace, size_t ws_bytes, int* info_host, void* stream);

/* The same SYRK step on the tensor cores (csrc/syrk_i8.cu): Cmat[Dpad,Dpad] -= Zt^T Zt for Zt double [Kpad,Dpad]
 * (Dpad a multiple of 128), FP64-equivalent through `slices` (3..7; 7 = 54 fractional bits) int8
 * Ozaki slices on tcgen05.mma kind::i8 with exact int32 accumulation in TMEM.  The row-major LOWER triangle is written.
 * vgg_ba_solve uses it with 7 slices; exposed for the parity tests and profiling. */
int vgg_syrk_ozaki_workspace_bytes(int Kpad, int Dpad, int slices, size_t* bytes);
int vgg_syrk_ozaki(int Kpad, int Dpad, const double* Zt, double* Cmat, int slices, void* workspace, size_t ws_bytes,
                   void* stream);
/* Whole Levenberg-Marquardt solve (Ceres trust-region semantics).  `trace` is a HOST array
 * [max_num_iterations, 8] (it, cost, candidate_cost, model_change, rho, radius, step_norm, flags) or NULL. */
int vgg_ba_solve(const vgg_ba_problem* prob, const vgg_ba_options* opt, void* workspace,
                 size_t ws_bytes, vgg_allreduce_fn allreduce, void* allreduce_user,
                 vgg_ba_summary* summary, double* trace, void* stream);
int vgg_ba_reduced_system_doubles(int S, int camera_model, int intr_mode, size_t* doubles);
int vgg_ba_fabric_doubles(int S, int camera_model, int intr_mode, size_t* doubles);
int vgg_ba_solve_fabric(const vgg_ba_problem* prob, const vgg_ba_options* opt, void* workspace,
                        size_t ws_bytes, vgg_allreduce_fn allreduce, void* allreduce_user,
                        const vgg_ba_fabric* fabric, vgg_ba_summary* summary, double* trace, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* Absolute-pose refinement: replaces the per-frame loop around pycolmap.pose_refinement        */
/* (vggsfm/utils/triangulation.py:260-479 refine_pose, :482-647 init_refine_pose).               */
/* ------------------------------------------------------------------------------------------- */

/* COLMAP AbsolutePoseRefinementOptions + the Ceres defaults behind it, plus the two pre-filters the
 * reference applies around the call: max_reproj_error > 0 ANDs the mask with (depth > 0 and squared
 * reprojection error <= max^2) at the input camera (triangulation.py:298-315); a frame is refined only
 * when its effective inlier count is > min_inliers (:386, :585). */
typedef struct vgg_pose_options {
  int32_t max_num_iterations;
  int32_t max_num_consecutive_invalid_steps;
  int32_t min_inliers;
  int32_t reserved;
  double function_tolerance, gradient_tolerance, parameter_tolerance;
  double initial_trust_region_radius, max_trust_region_radius, min_trust_region_radius;
  double min_relative_decrease, min_lm_diagonal, max_lm_diagonal;
  double loss_function_scale;   /* ceres::CauchyLoss scale */
  double max_reproj_error;      /* pixels; <= 0 disables the pre-filter */
} vgg_pose_options;

#define VGG_POSE_SKIPPED 6       /* frame_flags bit0 clear */
#define VGG_POSE_FEW_INLIERS 7   /* effective inliers <= min_inliers: pose left unchanged */

void vgg_pose_default_options(vgg_pose_options* opt);

/* One launch, one CTA per frame.  uv float [S,P,2] pixels; inlier uint8 [S,P]; frame_flags uint8 [S]
 * (bit0 refine this frame, bit1 refine_focal_length, bit2 refine_extra_params); points double [P,3]
 * (constant); poses [S,12] / intr [S,4] in/out.  Outputs: inlier_used uint8 [S,P] (the effective mask),
 * summary_d double [S,4] = (initial_cost, final_cost, final_radius, effective inliers), summary_i int32
 * [S,4] = (iterations, successful steps, termination VGG_BA_* / VGG_POSE_*, 0). */
int vgg_pose_refinement(int S, int P, int camera_model, const float* uv, const uint8_t* inlier,
                        const uint8_t* frame_flags, const double* points, double* poses, double* intr,
                        const vgg_pose_options* opt, uint8_t* inlier_used, double* summary_d, int32_t* summary_i,
                        void* stream);

/* ------------------------------------------------------------------------------------------- */
/* Triangulation side (float64, like the reference's real pipeline: models/triangulator.py:91) */
/* ------------------------------------------------------------------------------------------- */

/* triangulate_tracks / triangulate_tracks_single_chunk (vggsfm/utils/triangulation.py:677-956):
 * fused LORANSAC.  extrinsics [S,12]; tracks_normalized double [S,N,2]; track_vis/track_score float
 * [S,N] (score may be NULL); pairs int32 [H0,2] = the hypothesis frame pairs drawn on the host exactly
 * like triangulation.py:804-813 (CPU torch.randperm).  Outputs: points double [N,3], inlier_num
 * int64 [N], inlier_mask uint8 [N,S]. */
int vgg_tri_workspace_bytes(int S, int N, int H0, int lo_num, size_t* bytes);
int vgg_triangulate_tracks(int S, int N, const double* extrinsics, const double* tracks_normalized,
                           const float* track_vis, const float* track_score, const int32_t* pairs, int H0,
                           int lo_num, double max_angular_error_deg, double min_tri_angle_deg, double* out_points,
                           int64_t* out_inlier_num, uint8_t* out_inlier_mask, void* workspace, size_t ws_bytes,
                           void* stream);

/* triangulate_by_pair (triangulation.py:45-135): frame 0 against frames 1..S-1.  Outputs [S-1,N,3],
 * cheirality uint8 [S-1,N] (1 = in front of both), angle double [S-1,N] degrees.  workspace >= S*24 B. */
int vgg_triangulate_by_pair(int S, int N, const double* extrinsics, const double* tracks_normalized,
                            double* out_points, uint8_t* out_cheirality, double* out_angle_deg, void* workspace,
                            size_t ws_bytes, void* stream);

/* filter_all_points3D / _single_chunk (vggsfm/utils/triangulation_helpers.py:133-307).  points2d is
 * float or double [S,P,2]; intrinsics9 [S,9] row-major K; extra_params [S] SIMPLE_RADIAL k or NULL;
 * out_valid uint8 [P]; out_detail uint8 [S,P] or NULL (return_detail).  workspace >= S*24 B. */
int vgg_filter_points3d(int S, int P, const double* points3d, const void* points2d, int points2d_is_f64,
                        const double* extrinsics, const double* intrinsics9, const double* extra_params,
                        double max_reproj_error, double min_tri_angle_deg, int check_triangle, double hard_max,
                        uint8_t* out_valid, uint8_t* out_detail, void* workspace, size_t ws_bytes, void* stream);

/* project_3D_points / img_from_cam (triangulation_helpers.py:311-395): out_points2d [S,P,2] and/or
 * out_points_cam [S,3,P] (either may be NULL). */
int vgg_project_points(int S, int P, const double* points3d, const double* extrinsics, const double* intrinsics9,
                       const double* extra_params, double* out_points2d, double* out_points_cam, void* stream);

/* cam_from_img without distortion (triangulation_helpers.py:398-428): (uv - pp)/f in the input
 * precision (is_f64 selects float/double for tracks, focal2 [S,2], pp2 [S,2] and out). */
int vgg_normalize_tracks(int S, int N, const void* tracks, const void* focal2, const void* pp2, int is_f64, void* out,
                         void* stream);

/* iterative_undistortion (vggsfm/utils/distortion.py:27-99) for SIMPLE_RADIAL, with the reference's
 * semantics: damped Newton with a central-difference Jacobian and ONE global stop when the largest
 * squared step over all observations is < max_step_norm.  workspace >= 16 B. */
int vgg_undistort_simple_radial(int S, int N, const double* tracks_normalized, const double* extra_params,
                                int max_iterations, double max_step_norm, double rel_step_size, double* out,
                                int* iterations_run, void* workspace, size_t ws_bytes, void* stream);

/* pycolmap.absolute_pose_estimation for the frames refine_pose cannot refine (vggsfm/utils/triangulation.py:404-433:
 * estimate_focal_length = True, ransac.max_error = 12) and for the video runner's PnP alignment
 * (vggsfm/runners/video_runner.py:985-998): P3P + LO-RANSAC, batched over frames AND over COLMAP's 31 focal-length
 * factors (0.2 + 4.8 (i/30)^2) in one launch, on caller-drawn minimal samples (u_samples double [num_trials,3], uniform
 * in [0,1), mapped to the frame's usable points).  uv float [S,P,2] pixels, mask uint8 [S,P] usable observations,
 * frame_flags uint8 [S] (0 = skip the frame), points double [P,3], intr double [S,4] = f,cx,cy,k.
 * Out: pose_out double [S,12] (R|t, written for successful frames only), focal_out double [S] (prior focal x best
 * factor), num_inliers_out int32 [S] (0 = no model: the reference's `None`), inlier_out uint8 [S,P].
 * The non-linear refinement COLMAP runs afterwards is vgg_pose_refinement.  P <= ~9700 per call. */
int vgg_pnp_workspace_bytes(int S, int estimate_focal_length, size_t* bytes);
int vgg_absolute_pose_estimation(int S, int P, int camera_model, const float* uv, const uint8_t* mask,
                                 const uint8_t* frame_flags, const double* points, const double* intr,
                                 const double* u_samples, int num_trials, int estimate_focal_length, double max_error,
                                 double* pose_out, double* focal_out, int* num_inliers_out, uint8_t* inlier_out,
                                 void* workspace, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* Tracker correlation inner loop (float32 math on float or half feature pyramids)             */
/* ------------------------------------------------------------------------------------------- */

/* CorrBlock.__init__ (vggsfm/models/track_modules/blocks.py:339-361): feature pyramid by repeated
 * avg_pool2d(2,2), stored channels-last [BS,H_l,W_l,C] per level in `elem_size` bytes per element
 * (4 = float, 2 = half as under the reference's fp16 autocast, runners/runner.py:418).
 * fmaps_nchw is float [BS,C,H,W].  The half pyramid needs a float scratch (sizes from *_bytes). */
int vgg_corr_pyramid_bytes(int BS, int C, int H, int W, int num_levels, int elem_size, size_t* pyramid_bytes,
                           size_t* scratch_bytes);
int vgg_corr_build_pyramid(int BS, int C, int H, int W, int num_levels, const float* fmaps_nchw, int elem_size,
                           void* pyramid, void* scratch, void* stream);

/* CorrBlock.corr + CorrBlock.sample fused (blocks.py:363-416; border_padding=1 gives
 * EfficientCorrBlock.sample, :433-471).  targets float [BS,N,C], coords float [BS,N,2] (x,y) in level-0
 * pixels, out float [BS,N,num_levels*(2r+1)^2] with out[a*(2r+1)+b] sampled at (x+a-r, y+b-r). */
int vgg_corr_sample(int BS, int N, int C, int H, int W, int num_levels, int radius, const void* pyramid, int elem_size,
                    const float* targets, const float* coords, int border_padding, float* out, void* stream);

/* The same CorrBlock.corr + CorrBlock.sample for the coarse tracker's C = 128 maps ON THE TENSOR CORES
 * (csrc/corr_tc.cu: tcgen05.mma kind::f16 M=128 x N=256 x K=128 into TMEM, footprint extraction from TMEM in the
 * epilogue; the dense fp16 product of blocks.py:413 without ever storing the volume).  Zero padding only; map width a
 * power of two.  vgg_corr_tc_build turns the HALF channels-last pyramid of vgg_corr_build_pyramid into operand tile
 * images once per CorrBlock (tile_bytes from vgg_corr_tc_bytes); vgg_corr_tc_sample needs `target_bytes` of scratch for
 * the fp16 target tiles of the call.  Same targets / coords / out layout as vgg_corr_sample. */
int vgg_corr_tc_supported(int C, int H, int W, int num_levels, int radius);
int vgg_corr_tc_bytes(int BS, int C, int H, int W, int num_levels, int N, size_t* tile_bytes, size_t* target_bytes);
int vgg_corr_tc_build(int BS, int C, int H, int W, int num_levels, const void* pyramid_half, void* tiles, void* stream);
int vgg_corr_tc_sample(int BS, int N, int C, int H, int W, int num_levels, int radius, const void* tiles, const float* targets,
                       const float* coords, void* target_tiles, float* out, void* stream);

/* sample_features4d (vggsfm/models/utils.py:415-447; colour read-back at models/triangulator.py:324, query
 * features in the tracker): bilinear sampling, align_corners=True, border padding.  input float [B,C,H,W],
 * coords float [B,R,2] (x,y) pixels, out float [B,R,C]. */
int vgg_sample_features4d(int B, int C, int H, int W, int R, const float* input_nchw, const float* coords, float* out,
                          void* stream);

#ifdef __cplusplus
}
#endif
#endif
