/*
 * b200smpl.h -- C-ABI of the B200-native batched SMPL layer (libb200smpl.so).
 *
 * The reference has no FFI for this path: its boundary is a Python nn.Module
 * (`Python/Soccer/PlayerReconstruction/models/smpl_official.py:10-41`, a subclass of the
 * third-party `smplx.SMPL`).  Each entry point below states which reference interface it
 * replaces.  The Python host side (`soccerplayershapepose_b200/smpl.py`) binds these with
 * ctypes and re-creates the reference module's call surface on top (see INTEGRATION.md).
 *
 * Conventions
 *  - plain pointers + sizes, no torch / C++ types;
 *  - every tensor (inputs, outputs, workspace) is allocated and owned by the CALLER and passed
 *    as a raw DEVICE pointer, contiguous, row-major, fp32 unless noted; the library owns only
 *    the immutable pre-packed model buffers behind the handle;
 *  - all compute entry points are asynchronous on the given CUDA stream (`stream` is a
 *    `cudaStream_t` passed as `void*`; NULL = legacy default stream), never synchronise and
 *    never throw; return 0 on success or a negative B200SMPL_ERR_* code, with a message
 *    retrievable through b200smpl_last_error() (thread-local);
 *  - re-entrant across handles; a handle is bound to one device; no thread-local GPU state.
 *  - there is NO CPU fallback: without a CUDA device every compute call fails with
 *    B200SMPL_ERR_CUDA.
 */
#ifndef B200SMPL_H_
#define B200SMPL_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200SMPL_ABI_VERSION 1

#if defined(__GNUC__)
#define B200SMPL_API __attribute__((visibility("default")))
#else
#define B200SMPL_API
#endif

/* error codes */
#define B200SMPL_OK 0
#define B200SMPL_ERR_INVALID (-1)    /* bad argument / unsupported model */
#define B200SMPL_ERR_CUDA (-2)       /* CUDA runtime / driver error (message has details) */
#define B200SMPL_ERR_WORKSPACE (-3)  /* workspace too small */

/* arithmetic modes of the blend-shape contraction (BASELINE.json north_star: fp32 / bf16-GEMM) */
#define B200SMPL_MODE_FP32 0       /* tcgen05 bf16x3 error-compensated split, fp32 accumulate (~fp32 accuracy) */
#define B200SMPL_MODE_BF16 1       /* bf16-GEMM mode: forward blend with bf16 pose-corrective operands (template+shape
                                      still split-exact; positions within 1e-4 m); the gradient GEMM keeps the bf16x3
                                      split so that gradients stay within 1e-4 relative */
#define B200SMPL_MODE_FP32_SIMT 2  /* plain fp32 FFMA kernels (verification mode, slow) */
#define B200SMPL_MODE_BF16_FAST 3  /* MODE_BF16 forward + single-product bf16 gradient GEMM: grad_betas ~2e-3 relative,
                                      i.e. OUTSIDE the 1e-4 gradient tolerance; 9 % faster step */

typedef struct b200smpl_model b200smpl_model; /* opaque */

/*
 * Host-side description of an SMPL model; all pointers are HOST pointers, read during
 * b200smpl_model_create only.  Mirrors the buffers smplx.SMPL.__init__ registers
 * (v_template, shapedirs, posedirs, J_regressor, lbs_weights, parents) plus what
 * models/smpl_official.py:17-25 adds (J_regressor_extra/cocoplus/h36m, stacked) and the
 * smplx VertexJointSelector ids.
 */
typedef struct b200smpl_model_desc {
  int32_t num_verts;            /* V = 6890 */
  int32_t num_joints;           /* must be 24 */
  int32_t num_betas;            /* 10 (1..16) */
  int32_t num_vertex_joints;    /* 21 joints picked from vertices (may be 0) */
  int32_t num_regressed_joints; /* 45 = 9 + 19 + 17 joints regressed from vertices (may be 0) */
  int32_t reserved0;
  const float* v_template;          /* [V][3] */
  const float* shapedirs;           /* [V][3][num_betas] */
  const float* posedirs;            /* [207][V*3]  (smplx buffer layout, column = 3*v + k) */
  const float* J_regressor;         /* [24][V] */
  const float* lbs_weights;         /* [V][24], at most 4 non-zeros per row */
  const int64_t* parents;           /* [24], parents[0] = -1, parents[i] < i */
  const int64_t* vertex_joint_ids;  /* [num_vertex_joints] */
  const float* joint_regressors;    /* [num_regressed_joints][V] */
} b200smpl_model_desc;

/* sizes the caller needs to allocate outputs / workspace */
typedef struct b200smpl_model_info {
  int32_t num_verts;
  int32_t num_joints_out;      /* 24 + num_vertex_joints + num_regressed_joints (= 90) */
  int32_t num_betas;
  int32_t num_blend_rows;      /* 3V + 3 * (virtual joint rows) : rows of the packed blend operand */
  int32_t num_blend_rows_padded;
  int32_t feature_pitch;       /* K pitch of the packed operands (elements) */
  int32_t num_virtual_groups;
  int32_t device;              /* -1 for a host-only handle */
} b200smpl_model_info;

/*
 * Replaces: SMPL.__init__ (models/smpl_official.py:15-25 + smplx.SMPL.__init__): packs the
 * model for the GPU (bf16 split blend operand, 4-sparse skinning plan, joint terms) and uploads
 * it to `device`.  device = -1 builds a host-only handle (packing only; used by CPU tests).
 */
B200SMPL_API int b200smpl_model_create(const b200smpl_model_desc* desc, int device, b200smpl_model** out);
B200SMPL_API void b200smpl_model_destroy(b200smpl_model* m);
B200SMPL_API int b200smpl_model_get_info(const b200smpl_model* m, b200smpl_model_info* info);

/* Test hook: host copies of the packed arrays ("Wf", "Wb_hi", "Wb_lo", "W32", "vmeta", "vwts",
 * "term_ptr", "term_joint", "term_qrow", "term_c", "Jt", "Jsd"); valid until model_destroy. */
B200SMPL_API int b200smpl_model_debug_array(const b200smpl_model* m, const char* name, const void** data, size_t* bytes);

/* Bytes of caller-provided scratch needed by forward / backward for `batch` bodies.
 * slab_bodies = 0 lets the library pick the slab (bodies processed per L2-resident pass); a
 * request is rounded up to a multiple of 128 and capped at 40960 bodies (the widest slab the
 * forward GEMMs' work lists hold).  Results do not depend on the slab. */
/* Bytes of the optional "saved for backward" buffer (blend output + skinning transforms of the
 * whole batch, ~93 KB per body).  When forward writes it and backward receives it, the backward
 * skips the recomputation of the pose stage and of the blend GEMM. */
B200SMPL_API size_t b200smpl_saved_bytes(const b200smpl_model* m, int batch, int slab_bodies);
B200SMPL_API size_t b200smpl_forward_workspace_bytes(const b200smpl_model* m, int batch, int mode, int slab_bodies);
B200SMPL_API size_t b200smpl_backward_workspace_bytes(const b200smpl_model* m, int batch, int mode, int slab_bodies);

typedef struct b200smpl_forward_args {
  int32_t batch;               /* B >= 1 */
  int32_t mode;                /* B200SMPL_MODE_* */
  int32_t pose_is_axis_angle;  /* 1: pose is [B][72] axis-angle (smplx pose2rot=True); 0: [B][24][3][3] */
  int32_t slab_bodies;         /* 0 = auto */
  const float* betas;          /* [B][num_betas] */
  const float* pose;           /* [B][24][9] rotation matrices (row-major) or [B][72] */
  const float* transl;         /* [B][3] or NULL */
  const float* cam;            /* [B][3] weak-perspective [s,tx,ty] or NULL (enables joints2d) */
  float* vertices;             /* out [B][V][3], or NULL for the joints-only path */
  float* joints;               /* out [B][num_joints_out][3] */
  float* joints2d;             /* out [B][num_joints_out][2] = s*(x+tx), s*(y+ty); NULL if cam is NULL */
  void* workspace;
  size_t workspace_bytes;
  void* saved;                 /* out, optional: b200smpl_saved_bytes(B, slab) bytes kept for backward; a joints-only
                                  call (vertices == NULL) fills only the joint rows: pass grad_vertices = NULL to
                                  the backward that receives it */
  size_t saved_bytes;
} b200smpl_forward_args;

/*
 * Replaces: SMPL.forward (models/smpl_official.py:27-41 -> smplx.SMPL.forward -> smplx.lbs.lbs,
 * VertexJointSelector, 3x vertices2joints) and, when cam != NULL, orthographic_project_torch
 * (utils/cam_utils.py:5-26) applied to the joints.
 */
B200SMPL_API int b200smpl_forward(const b200smpl_model* m, const b200smpl_forward_args* args, void* stream);

typedef struct b200smpl_backward_args {
  int32_t batch;
  int32_t mode;
  int32_t pose_is_axis_angle;
  int32_t slab_bodies;
  const float* betas;            /* forward inputs again (needed by the chain backward and for recomputation) */
  const float* pose;
  const float* transl;           /* may be NULL */
  const float* cam;              /* may be NULL */
  const float* joints;           /* forward output [B][NJ][3]; required only if grad_joints2d != NULL */
  const float* grad_vertices;    /* [B][V][3] or NULL */
  const float* grad_joints;      /* [B][NJ][3] or NULL */
  const float* grad_joints2d;    /* [B][NJ][2] or NULL */
  float* grad_betas;             /* out [B][num_betas] */
  float* grad_pose;              /* out, same layout as pose */
  float* grad_transl;            /* out [B][3] or NULL */
  float* grad_cam;               /* out [B][3] or NULL */
  void* workspace;
  size_t workspace_bytes;
  const void* saved;             /* optional: what forward wrote with the same batch / slab_bodies; NULL = recompute */
  size_t saved_bytes;
} b200smpl_backward_args;

/*
 * Replaces: torch autograd over the reference's op graph (loss.backward() at
 * player_recon.py:1280 re-entering smplx.lbs).  Hand-written backward of every forward piece.
 */
B200SMPL_API int b200smpl_backward(const b200smpl_model* m, const b200smpl_backward_args* args, void* stream);

/* ---- small in-tree helpers of the path, forward + hand-written backward -------------------- */

/* smplx.lbs.batch_rodrigues (called directly by the reference at player_recon.py:201,655, hmr.py:207, and inside
 * smplx.lbs.lbs when pose2rot=True): rot_vecs [n][3] -> R [n][3][3], theta = ||r + 1e-8|| as smplx computes it */
B200SMPL_API int b200smpl_batch_rodrigues(const float* rot_vecs, float* rotmats, int64_t n, void* stream);
B200SMPL_API int b200smpl_batch_rodrigues_backward(const float* rot_vecs, const float* grad_rotmats, float* grad_rot_vecs,
                                                   int64_t n, void* stream);

/* utils/rigid_transform_utils.py:27-41 rot6d_to_rotmat: x [n][3][2] -> R [n][3][3] (columns b1,b2,b3) */
B200SMPL_API int b200smpl_rot6d_to_rotmat(const float* x6, float* rotmats, int64_t n, void* stream);
B200SMPL_API int b200smpl_rot6d_to_rotmat_backward(const float* x6, const float* grad_rotmats, float* grad_x6, int64_t n,
                                      void* stream);

/* utils/cam_utils.py:5-26 orthographic_project_torch: points [B][N][3], cam [B][3] -> [B][N][2].
 * pixel_wh > 0 additionally applies utils/joints2d_utils.py:5-10 undo_keypoint_normalisation. */
B200SMPL_API int b200smpl_orthographic_project(const float* points, const float* cam, float* out, int batch, int n,
                                  float pixel_wh, void* stream);
B200SMPL_API int b200smpl_orthographic_project_backward(const float* points, const float* cam, const float* grad_out,
                                           float* grad_points, float* grad_cam, int batch, int n, float pixel_wh,
                                           void* stream);

/* utils/cam_utils.py:54-85 perspective_project_torch with K = [[f,0,c],[0,f,c],[0,0,1]], c = img_wh/2:
 * points [B][N][3], rotation [B][3][3], translation [B][3] -> [B][N][2] */
B200SMPL_API int b200smpl_perspective_project(const float* points, const float* rotation, const float* translation, float* out,
                                 int batch, int n, float focal_length, float img_wh, void* stream);
B200SMPL_API int b200smpl_perspective_project_backward(const float* points, const float* rotation, const float* translation,
                                          const float* grad_out, float* grad_points, float* grad_rotation,
                                          float* grad_translation, int batch, int n, float focal_length,
                                          float img_wh, void* stream);

/* the same with an explicit intrinsics matrix (the cam_K argument of utils/cam_utils.py:54-85): cam_K [B][3][3]
 * (cam_K_batched != 0) or one [3][3] shared by the batch; out = rows 0 and 1 of K . (X'/z).  No gradient for cam_K. */
B200SMPL_API int b200smpl_perspective_project_camk(const float* points, const float* rotation, const float* translation,
                                                   const float* cam_K, int cam_K_batched, float* out, int batch, int n,
                                                   void* stream);
B200SMPL_API int b200smpl_perspective_project_camk_backward(const float* points, const float* rotation,
                                                            const float* translation, const float* cam_K,
                                                            int cam_K_batched, const float* grad_out, float* grad_points,
                                                            float* grad_rotation, float* grad_translation, int batch,
                                                            int n, void* stream);

/*
 * Fused joints2D loss term (losses/multi_task_loss.py:97-113 on top of player_recon.py:1217-1221):
 *   j2d = undo_keypoint_normalisation(orthographic(joints, cam)[:, map], proj_wh)
 *   loss = mean_{visible}( (2*j2d/norm_wh - 1  -  (2*label/norm_wh - 1))^2 ) * exp(-log_var) + log_var
 * joints [B][NJ][3], cam [B][3], joint_map [nmap] (device int32), label [B][nmap][2] pixels,
 * vis [B][nmap] uint8 or NULL, loss: device buffer of 2 floats zeroed by the caller ([0] receives
 * the loss, [1] is scratch for the visible-pair count),
 * grad_joints [B][NJ][3] and grad_cam [B][3] written (d loss / d .) when non-NULL.
 */
B200SMPL_API int b200smpl_joints2d_loss(const float* joints, const float* cam, const int32_t* joint_map, const float* label,
                           const uint8_t* vis, int batch, int num_joints, int nmap, float proj_wh, float norm_wh,
                           float log_var, float* loss, float* grad_joints, float* grad_cam, void* stream);

/*
 * Batched per-player fitting loop -- replaces the body of the reference's single_view_optimization
 * (player_recon.py:1172-1294: Adam over global_orient / body pose without hands and feet / cam / betas on the
 * joints2D loss, best iterate kept) for a batch of independent players.  One iteration is
 *   b200smpl_forward (joints only) -> b200smpl_fit_loss -> b200smpl_backward -> b200smpl_fit_mark_best ->
 *   b200smpl_fit_adam_step per parameter tensor
 * and is CUDA-graph capturable: the step counter and the "improved" flags live in device memory.
 *
 * fit_loss: loss_per_body[b] = mean over the player's visible (joint, xy) pairs of the squared normalised
 *   reprojection error (cam_utils.py:5-26 -> joints2d_utils.py:5-10 -> multi_task_loss.py:97-113 for ONE player)
 *   * exp(-log_var) + log_var + shape_weight * mean(betas^2)   (multi_task_loss.py:120-124 against zeros);
 *   grad_joints [B][NJ][3], grad_cam [B][3], grad_betas [B][nb] (shape term only; may be NULL) are written.
 * fit_mark_best: improved[b] = loss < best_loss (best_loss, best_iter updated); step[1] = step[0] + 1.
 * fit_adam_step: params [B][cols]; rows flagged improved are first copied to best_params (the parameters that
 *   produced this iteration's loss, player_recon.py:1258-1262), then torch.optim.Adam's update with the gradient
 *   grad (+ grad_extra) is applied to every column not marked in frozen_cols [cols] (may be NULL).  step is the
 *   2-int device counter shared with fit_mark_best; the call of an iteration's last tensor passes commit_step=1.
 */
B200SMPL_API int b200smpl_fit_loss(const float* joints, const float* cam, const int32_t* joint_map, const float* label,
                      const uint8_t* vis, const float* betas, int batch, int num_joints, int nmap, int num_betas,
                      float proj_wh, float norm_wh, float log_var, float shape_weight, float* loss_per_body,
                      float* grad_joints, float* grad_cam, float* grad_betas, void* stream);
B200SMPL_API int b200smpl_fit_mark_best(const float* loss_per_body, float* best_loss, int32_t* best_iter, uint8_t* improved,
                           int32_t* step, int batch, void* stream);
B200SMPL_API int b200smpl_fit_adam_step(float* params, const float* grad, const float* grad_extra, float* exp_avg,
                           float* exp_avg_sq, float* best_params, const uint8_t* improved, const uint8_t* frozen_cols,
                           int32_t* step, int commit_step, int batch, int cols, float lr, float beta1, float beta2,
                           float eps, void* stream);

/* fit_update: fit_mark_best and the fit_adam_step of up to B200SMPL_FIT_MAX_GROUPS parameter tensors in one launch
 * (the per-iteration tail of the fitting loop, player_recon.py:1254-1266 + 1281).  The step counter is double-buffered:
 * the call reads step[parity] and writes step[1 - parity]; the caller alternates the parity from a zeroed counter.
 * first_loss (may be NULL) receives the loss of iteration 1. */
#define B200SMPL_FIT_MAX_GROUPS 4
typedef struct b200smpl_fit_group {
  float* params;              /* [batch][cols] */
  const float* grad;          /* [batch][cols] */
  const float* grad_extra;    /* [batch][cols] added to grad, or NULL */
  float* exp_avg;             /* Adam first moment */
  float* exp_avg_sq;          /* Adam second moment */
  float* best_params;         /* rows of improved bodies are copied here before the update */
  const uint8_t* frozen_cols; /* [cols] 1 = never updated, or NULL */
  int32_t cols;
} b200smpl_fit_group;
B200SMPL_API int b200smpl_fit_update(const b200smpl_fit_group* groups, int ngroups, const float* loss_per_body,
                                     float* best_loss, int32_t* best_iter, float* first_loss, int32_t* step, int parity,
                                     int batch, float lr, float beta1, float beta2, float eps, void* stream);

/*
 * Fused multi-task loss of the regressor training step -- replaces HomoscedasticUncertaintyWeightedMultiTaskLoss
 * (losses/multi_task_loss.py:92-130, without its silhouette term; see b200smpl_silhouette_loss) as called at PyTorch3DTest.py:1072-1106:
 *   loss = sum over the present terms of  mean((pred - label)^2) * exp(-log_var_t) + log_var_t
 * terms t = 0 vertices, 1 2D joints (orthographic_project_torch(joints, cam)[:, map2d] -> undo_keypoint_normalisation
 * (proj_wh) -> both sides 2x/norm_wh - 1, optional vis mask over (body, joint) pairs), 2 3D joints (joints[:, map3d]),
 * 3 shape parameters, 4 pose rotation matrices.  A term is present when its prediction pointer (map pointer for the
 * joint terms) is non-NULL.  All pointers are DEVICE pointers; log_var [5] and the upstream gradient are read on the
 * device, so forward and backward are CUDA-graph capturable.
 *   forward : out[0] = loss, out[1..5] = weighted parts, out[6..10] = d loss / d log_var_t; fills scratch
 *   backward: gradients of  grad_loss[0] * loss  (grad_loss NULL = 1) w.r.t. vertices / joints [B][NJ][3] (both joint
 *             terms accumulated) / cam / shape / pose; any output may be NULL.  Needs the scratch of the forward.
 */
typedef struct b200smpl_multitask_loss_args {
  int32_t batch, num_verts, num_joints, nmap2d, nmap3d, num_betas, pose_cols, reserved0;
  float proj_wh, norm_wh;         /* 512, 256 in the reference (player_recon.py:1220, config.REGRESSOR_IMG_WH) */
  const float* verts;             /* [B][V][3] or NULL */
  const float* verts_label;
  const float* joints;            /* [B][NJ][3] */
  const float* cam;               /* [B][3] */
  const int32_t* map2d;           /* [nmap2d] or NULL */
  const float* label2d;           /* [B][nmap2d][2] pixels */
  const uint8_t* vis;             /* [B][nmap2d] or NULL */
  const int32_t* map3d;           /* [nmap3d] or NULL */
  const float* label3d;           /* [B][nmap3d][3] */
  const float* shape;             /* [B][num_betas] or NULL */
  const float* shape_label;
  const float* pose;              /* [B][pose_cols] or NULL */
  const float* pose_label;
  const float* log_var;           /* [5] */
  float* scratch;                 /* [16] floats, written by the forward, read by the backward */
} b200smpl_multitask_loss_args;
B200SMPL_API int b200smpl_multitask_loss(const b200smpl_multitask_loss_args* args, float* out, void* stream);
B200SMPL_API int b200smpl_multitask_loss_backward(const b200smpl_multitask_loss_args* args, const float* grad_loss,
                                                  float* grad_verts, float* grad_joints, float* grad_cam,
                                                  float* grad_shape, float* grad_pose, void* stream);

/*
 * Batched silhouette rasteriser of posed meshes -- replaces the reference's neural-renderer call
 * nmr(vertices, faces, t) (player_recon.py:1226-1229, 1084-1087) and pytorch3d's SoftSilhouetteShader
 * (PyTorch3DTest.py:64-238).  Definition (DESIGN.md section 11):
 *   camera   R = I, t = cam_t[b], K = [[f,0,S/2],[0,f,S/2],[0,0,1]] at S = img_wh:
 *            u = f (x+tx)/(z+tz) + S/2, v = f (y+ty)/(z+tz) + S/2; alpha[b][i][j] is the pixel centred at
 *            (u, v) = (j + 0.5, i + 0.5), no vertical flip;
 *   dropped  faces with a vertex at z+tz <= 1e-3 or |projected signed area| < 1e-8 px^2; winding is ignored;
 *   hard     sigma == 0: 1 where the pixel centre is inside or on the boundary of a kept face, else 0;
 *   soft     sigma  > 0 (px^2): D_f = sigmoid(+d^2/sigma) inside, sigmoid(-d^2/sigma) outside, d = distance to the
 *            face's nearest edge segment; an outside face with d^2 > sigma ln(1/1e-4 - 1) contributes nothing;
 *            alpha = 1 - prod_f (1 - D_f).
 * vertices [B][V][3], cam_t [B][3], faces [F][3] device int32 (V <= 65535; the projected vertices, a face list and,
 * for the backward, a per-vertex gradient accumulator must fit in one CTA's shared memory: SMPL needs 193 KB).
 * The backward is the exact derivative w.r.t. vertices and cam_t; the hard mode has none (B200SMPL_ERR_INVALID).
 * grad_vertices [B][V][3] and grad_t [B][3] are written, not accumulated.
 * silhouette_loss: loss_per_body[b] += weight * mean over the S^2 pixels of (alpha - target)^2 (target [B][S][S]
 * uint8, non-zero = inside), with the gradient of that term written to grad_vertices / grad_t; it never writes the
 * image.  The call adds into loss_per_body so that it can follow b200smpl_fit_loss on the same buffer.
 * No workspace is needed at present (workspace_bytes returns 0; the fields may be NULL / 0).
 */
typedef struct b200smpl_silhouette_args {
  int32_t batch, num_verts, num_faces, img_wh;
  float focal_length, sigma;
  const float* vertices;         /* [B][V][3] */
  const float* cam_t;            /* [B][3] camera translation */
  const int32_t* faces;          /* [F][3] */
  void* workspace;
  size_t workspace_bytes;
} b200smpl_silhouette_args;
B200SMPL_API size_t b200smpl_silhouette_workspace_bytes(const b200smpl_silhouette_args* args);
B200SMPL_API int b200smpl_silhouette_render(const b200smpl_silhouette_args* args, float* alpha, void* stream);
B200SMPL_API int b200smpl_silhouette_render_backward(const b200smpl_silhouette_args* args, const float* grad_alpha,
                                                     float* grad_vertices, float* grad_t, void* stream);
B200SMPL_API int b200smpl_silhouette_loss(const b200smpl_silhouette_args* args, const uint8_t* target, float weight,
                                          float* loss_per_body, float* grad_vertices, float* grad_t, void* stream);

/* Test hook (host arithmetic only, no device): the cluster work list of the forward blend GEMM for `body_tiles`
 * 128-body tiles x `row_tiles` 128-row tiles on a device with `num_sms` SMs.  Writes (body-tile pair, first row-tile
 * pair, end row-tile pair) per cluster into out[3 * capacity]; returns the number of clusters or -1. */
B200SMPL_API int b200smpl_debug_fwd_gemm_worklist(int body_tiles, int row_tiles, int num_sms, uint16_t* out, int capacity);

B200SMPL_API const char* b200smpl_last_error(void);
B200SMPL_API int b200smpl_abi_version(void);

/* Per-kernel device timing for bench.py's roofline: while enabled (enable != 0) every kernel launch
 * is bracketed by CUDA events on its own stream.  b200smpl_timing_report synchronises those events and
 * writes one line per kernel name, "name launches total_ms\n", into buf (NUL-terminated, truncated to
 * cap), clears the records and returns the number of bytes needed. */
B200SMPL_API void b200smpl_timing_enable(int enable);
B200SMPL_API size_t b200smpl_timing_report(char* buf, size_t cap);

/* number of kernels this library has launched in the calling process (bench.py gpu_launches) */
B200SMPL_API int64_t b200smpl_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* B200SMPL_H_ */
