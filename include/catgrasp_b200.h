/*
 * catgrasp_b200.h -- C ABI of libcatgrasp_b200.so (sm_100a).
 *
 * This is the drop-in boundary for CaTGrasp's per-scene grasp-scoring hot
 * path.  Every entry point is `extern "C"`, takes plain pointers and sizes,
 * returns an int status (0 = ok, negative = CG_E*), and never calls exit().
 * Each entry cites the reference interface (file:line under the reference
 * checkout) that it replaces.
 *
 * Pointer conventions
 *   *_host : the function takes HOST buffers, performs H2D, compute and D2H
 *            itself on the context stream and returns after the result is in
 *            the host output buffer (the reference-facing, blocking call).
 *   *_dev  : all data pointers are DEVICE pointers owned by the caller
 *            (e.g. torch allocations); the call enqueues work on the context
 *            stream and returns without synchronising.
 * Row-major everywhere.  Poses are 4x4 row-major.
 */
#ifndef CATGRASP_B200_H
#define CATGRASP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes ------------------------------------------------------ */
#define CG_OK            0
#define CG_EINVAL       -1   /* bad argument / shape (reference: printf+exit(1),
                                my_cpp/collision_manager.cpp:17-27,57-61)     */
#define CG_ECUDA        -2   /* CUDA runtime error, see cg_last_error()       */
#define CG_ENOMEM       -3
#define CG_EUNSUPPORTED -4

typedef struct cg_ctx cg_ctx;   /* one per device; owns stream + workspace    */
typedef struct cg_net cg_net;   /* folded PointNetCls / PointNetSeg weights   */
typedef struct cg_sdf cg_sdf;   /* one Sdf3D grid resident in HBM             */

/* ---- context ----------------------------------------------------------- */
int         cg_ctx_create(int device, cg_ctx **out);
void        cg_ctx_destroy(cg_ctx *ctx);
/* Enqueue on a caller-owned cudaStream_t (passed as void*).  NULL means the
 * CUDA legacy default stream (stream 0), NOT the context's own stream; a new
 * context starts on its own non-blocking stream (cg_ctx_use_own_stream).      */
int         cg_ctx_set_stream(cg_ctx *ctx, void *cuda_stream);
int         cg_ctx_use_own_stream(cg_ctx *ctx);
int         cg_ctx_synchronize(cg_ctx *ctx);
const char *cg_last_error(cg_ctx *ctx);
const char *cg_version(void);
/* number of kernels this library launched on ctx since creation / reset.   */
int64_t     cg_ctx_launch_count(cg_ctx *ctx);
void        cg_ctx_reset_launch_count(cg_ctx *ctx);
/* GEMM engine of the fused shared-MLP "trunk":
 *   0 = fp32 SIMT (exact-order reference engine)
 *   1 = tcgen05, bf16 hi/lo x hi/lo, 3 passes (near-fp32: |dprob| ~ 1e-7)
 *   2 = tcgen05, 128->1024 layer with fp16 hi/lo activations x one fp16 weight
 *       term, 2 passes (|dprob| ~ 2e-6 vs the 1e-4 tolerance)
 *   3 = persistent tcgen05 kernel (one CTA per SM looping over candidates), the
 *       128->1024 layer as ONE fp16 x fp16 pass (|dprob| ~ 4e-6)            [default]
 *   (2 and 3 fall back to 1 for a net whose folded weights exceed the fp16 range) */
int         cg_ctx_set_engine(cg_ctx *ctx, int engine);
int         cg_ctx_get_engine(cg_ctx *ctx);
/* Engines 2/3 clamp the 128->1024 layer's inputs to the fp16 range (65504).
 * *out = 1 if a clamp happened on this context since the previous call (the
 * flag is cleared); the caller should then re-run on engine 1.  Synchronises
 * the context's stream.                                                      */
int         cg_ctx_fp16_overflow(cg_ctx *ctx, int *out);
/* Diagnostic: exercises the TMEM fragment layout the engine-3 max epilogue
 * relies on; out_host receives 768 floats (see tests/test_gpu_parity.py).    */
int         cg_tmem_layout_selftest(cg_ctx *ctx, float *out_host);
/* Optional in-stream timing of the dominant kernel (the fused shared-MLP+max
 * "trunk"): when enabled every trunk launch is bracketed by a CUDA event pair
 * on the launching stream; cg_ctx_profile_read() synchronises those events and
 * returns the summed duration and the launch count, then clears the list.   */
int         cg_ctx_profile(cg_ctx *ctx, int enable);
int         cg_ctx_profile_read(cg_ctx *ctx, double *ms_total, int64_t *launches);

/* ---- networks ----------------------------------------------------------
 * Replaces: pointnet2.py:275-299 (PointNetCls), :302-329 (PointNetSeg),
 * loaded through Utils.py:135-148 (load_model).  The host side folds every
 * BatchNorm into the preceding conv/linear and packs fp32 weights in the
 * order documented in catgrasp_b200/weights.py; `blob` is that packing.
 *   kind: 0 = PointNetCls(n_in=6, n_out), 1 = PointNetSeg(n_in=6, n_out)     */
#define CG_NET_CLS 0
#define CG_NET_SEG 1
int  cg_net_create(cg_ctx *ctx, int kind, int n_out,
                   const float *blob_host, size_t blob_floats, cg_net **out);
void cg_net_destroy(cg_net *net);
size_t cg_net_blob_floats(int kind, int n_out);

/* Grasp-Q forward over B candidates.
 * Replaces: predicter.py:67-94 (GraspPredicter.predict_batch) incl. the
 * per-candidate GraspDataset.transform (dataset_grasp.py:63-91) which is
 * fused into the first kernel: for candidate b, point n
 *     id   = ids[b*N+n]                       (host-drawn numpy RNG indices)
 *     xyz  = inv(pose_b)     * cloud_xyz[id]  (float64, like the reference)
 *     nrm  = inv(pose_b[:3,:3]) * cloud_nrm[id]
 *     in6  = ([xyz,nrm] - mean) / (std + 1e-15)   (if mean/std != NULL)
 * then PointNetCls forward + softmax in fp32.
 *   cloud_xyz, cloud_nrm : (M,3) float64      poses : (B,4,4) float64
 *   ids : (B,N) int32 in [0,M)                mean,std : (6,) float64 or NULL
 *   out_probs : (B,n_out) float32             out_label : (B,) int32 or NULL
 */
int cg_graspq_forward_host(cg_net *net,
                           const double *cloud_xyz, const double *cloud_nrm, int M,
                           const double *poses, int B,
                           const int32_t *ids, int N,
                           const double *mean, const double *std,
                           float *out_probs, int32_t *out_label);
int cg_graspq_forward_dev(cg_net *net,
                          const double *cloud_xyz, const double *cloud_nrm, int M,
                          const double *poses, int B,
                          const int32_t *ids, int N,
                          const double *mean, const double *std,
                          float *out_probs, int32_t *out_label);

/* The per-candidate point-subset draw of GraspDataset.transform
 * (dataset_grasp.py:72-73: np.random.choice(np.arange(M), size=n_pts,
 * replace=(M < n_pts)) from the GLOBAL legacy numpy generator, once per
 * candidate, in candidate order).
 *
 * cg_host_legacy_choice (HOST function, no GPU work): the same draw, bit for
 * bit, without the Python-level call per candidate.  key[624] / *pos are the
 * MT19937 state of np.random.get_state() (fields 1 and 2); both are advanced
 * exactly as numpy would advance them, so np.random.set_state() afterwards
 * leaves the host program on the reference's random stream.  The stream walk
 * is sequential (AVX-512 / AVX2 / scalar, picked at load time); the
 * permutations are replayed on `nthreads` host threads (<= 0: one per core,
 * at most 12).  out: (count, n_pts) int32.
 * cg_host_rng_isa(level) caps the instruction set (0 scalar, 1 AVX2, 2 AVX-512,
 * -1 best available) and returns the level in use -- a test hook.
 *
 * cg_draw_ids_dev (opt-in, NOT the reference's numbers): a counter-based draw
 * on the device with the same distribution -- n_pts distinct uniform indices
 * (keyed Feistel permutation of [0,M), cycle-walked) when M >= n_pts, n_pts
 * independent uniform indices when M < n_pts.  Candidate b uses the key
 * (seed, first_candidate + b), so shards of one candidate list draw the same
 * subsets as the unsharded call.  out_ids: (count, n_pts) int32 on device.   */
int cg_host_legacy_choice(uint32_t *key, int32_t *pos, int64_t M, int32_t n_pts,
                          int32_t count, int32_t *out, int32_t nthreads);
/* advance the generator over `count` candidates without producing their indices (sharded scoring) */
int cg_host_legacy_skip(uint32_t *key, int32_t *pos, int64_t M, int32_t n_pts, int32_t count);
int cg_host_rng_isa(int level);
int cg_draw_ids_dev(cg_ctx *ctx, int M, int n_pts, int count, uint64_t seed,
                    int64_t first_candidate, int32_t *out_ids);

/* PointNetCls / PointNetSeg forward on an already materialised input tensor
 * x : (B,N,6) float32 (device).  Replaces pointnet2.py:289-299 / :316-329.
 *   cls: out_logits (B,n_out) and/or out_probs (B,n_out) (either may be NULL)
 *   seg: out_logits (B,N,n_out) float32                                     */
int cg_cls_forward_dev(cg_net *net, const float *x, int B, int N,
                       float *out_logits, float *out_probs);
int cg_seg_forward_dev(cg_net *net, const float *x, int B, int N,
                       float *out_logits);
/* NUNOCS post-processing, predicter.py:144-150: logits (P, 3*bins) ->
 * coords (P,3) = argmax*(1/bins) - 0.5 and conf_z (P,) = softmax prob of the
 * z-axis argmax bin.  Fused variant of cg_seg_forward for B=1.              */
int cg_nunocs_forward_host(cg_net *net, const float *x_host, int N, int bins,
                           float *out_coords, float *out_conf_z, int32_t *out_bins);
int cg_nunocs_forward_dev(cg_net *net, const float *x, int N, int bins,
                          float *out_coords, float *out_conf_z, int32_t *out_bins);

/* ---- SDF grid ----------------------------------------------------------
 * Replaces: meshpy/meshpy/sdf.py:217-289 (Sdf3D), sdf_file.py:59-87.
 * grid is data[i][j][k] row-major (k fastest) float32; grid coordinate of a
 * point x (SDF frame) is (x - origin) / resolution (sdf.py:252-264).        */
int  cg_sdf_create(cg_ctx *ctx, const float *grid_host, int nx, int ny, int nz,
                   const float origin[3], float resolution, cg_sdf **out);
void cg_sdf_destroy(cg_sdf *sdf);
/* Point-wise signed distance lookups at GRID coordinates (P,3) float32.
 *   mode 0: trilinear, sdf.py:292-343 (_signed_distance)
 *   mode 1: nearest cell with clamp, sdf.py:345-359 (_signed_distance_batch) */
#define CG_SDF_TRILINEAR 0
#define CG_SDF_NEAREST   1
int cg_sdf_lookup_dev(cg_sdf *sdf, const float *grid_coords, int P, int mode,
                      float *out_sd);

/* ---- collision filter --------------------------------------------------
 * Replaces: my_cpp/common.cpp:156-321 (filterGraspPose) with the FCL
 * mesh-vs-octree test (collision_manager.cpp:93-111) substituted by the
 * gripper-SDF predicate of sdf.py:377-389 (is_any_points_inside, nearest
 * mode) or its trilinear form (sdf.py:292-343).  IK (common.cpp:214-226) is
 * NOT evaluated here (see INTEGRATION.md): pass filter results to the host
 * ikfast stage.
 *   grasp_poses (G,4,4), symmetry_tfs (S,4,4), the five 4x4 matrices:
 *       float32 row-major (the reference narrows float64 -> float at the
 *       pybind boundary, common.h:51,60).
 *   open_pts (P1,3), enclosed_pts (P2,3): float32 camera-frame points
 *       (gripper_collision_pts / gripper_enclosed_collision_pts).
 *   Outputs are indexed by pair q = i*S + j, i.e. DETERMINISTIC order
 *   (the reference's is thread-arrival order, common.cpp:303-313):
 *   out_status[q] : 0 accepted, 1 rejected by approach direction,
 *                   3 rejected by collision (2 is reserved for IK)
 *   out_offset[q] : index 0..4 of the winning lateral offset
 *                   (0,+1mm,-1mm,+2mm,-2mm; common.cpp:255-262), -1 if none
 *   out_poses[q]  : (4,4) float32 grasp_in_cam shifted by the winning offset,
 *                   all-zero when rejected (common.cpp:289-293)              */
#define CG_ST_ACCEPT    0
#define CG_ST_REJ_DIR   1
#define CG_ST_REJ_IK    2
#define CG_ST_REJ_COLL  3   /* collision (with split_coll_status and no pose adjustment: the OPEN gripper hits the object) */
#define CG_ST_REJ_COLL_ENCL 4   /* split_coll_status only: the open gripper is free, the ENCLOSED gripper hits the background */
typedef struct cg_filter_params {
  float nocs_pose[16];
  float canonical_to_nocs[16];
  float gripper_in_grasp[16];
  int   filter_approach_dir_face_camera;
  int   adjust_collision_pose;
  int   sdf_mode;          /* CG_SDF_TRILINEAR or CG_SDF_NEAREST */
  float sdf_margin;        /* a scene point collides iff sd < sdf_margin (metres).  0 = the SDF predicate of
                              meshpy/sdf.py:377-389 (point inside the gripper solid).  octo_resolution*sqrt(3)/2 makes
                              the verdict conservative w.r.t. the reference's mesh-vs-voxel test
                              (my_cpp/collision_manager.cpp:93-111): every occupied voxel cube of side
                              octo_resolution that can touch the gripper surface has its generating point within
                              that distance of the surface.                                                        */
  int   split_coll_status; /* != 0 and adjust_collision_pose == 0: report which of the reference's two tests rejected a
                              pose (CG_ST_REJ_COLL = open gripper vs object points, common.cpp:231-238;
                              CG_ST_REJ_COLL_ENCL = enclosed gripper vs background, :241-248) -- the verbose counters
                              n_open_gripper_rej / n_close_gripper_rej.  Costs the reference's scan order (open first)
                              instead of the faster background-sample-first order.  With pose adjustment the reference
                              itself counts every collision rejection as "open" (:290-294): always CG_ST_REJ_COLL.     */
} cg_filter_params;

int cg_filter_grasp_pose_host(cg_ctx *ctx, const cg_filter_params *prm,
                              const float *grasp_poses, int G,
                              const float *symmetry_tfs, int S,
                              cg_sdf *sdf_open, const float *open_pts, int P1,
                              cg_sdf *sdf_enclosed, const float *enclosed_pts, int P2,
                              uint8_t *out_status, int8_t *out_offset, float *out_poses);
int cg_filter_grasp_pose_dev(cg_ctx *ctx, const cg_filter_params *prm,
                             const float *grasp_poses, int G,
                             const float *symmetry_tfs, int S,
                             cg_sdf *sdf_open, const float *open_pts, int P1,
                             cg_sdf *sdf_enclosed, const float *enclosed_pts, int P2,
                             uint8_t *out_status, int8_t *out_offset, float *out_poses);

/* ---- collision filter, mesh-vs-voxel predicate ------------------------------
 * The reference's own geometry test (my_cpp/collision_manager.cpp:15-111: FCL
 * BVH of the gripper mesh vs an octomap OcTree of the points), restated in
 * oracle/mesh_voxel_ref.py and computed here bit for bit:
 *   occupied voxel  = unique key floor(double(x) * (1.0 / res)) per axis with
 *                     res = double(float32 resolution); keys outside
 *                     [-32768, 32768) are dropped (octomap coordToKeyChecked);
 *                     the cube [key*res, (key+1)*res] per axis;
 *   posed mesh      = float32 gripper_in_cam of cg_filter_grasp_pose_* widened to
 *                     double, Vc = ((R0*vx + R1*vy) + R2*vz) + t, no contraction;
 *   collision       = some cube overlaps some posed triangle under the 13-axis
 *                     separating-axis test in double (touching collides).
 *
 * cg_mesh (registerMesh): the (nv,3) float32 vertices and (nf,3) int32 faces in
 * the gripper frame plus a uniform grid of cubic cells over their bounding box
 * with CSR lists of the triangles meeting each (closed) cell, built on the host.
 * Cell-size rule: edge = max(cbrt(box volume / (2 nf)), extent / 1023), where
 * the box volume uses each extent clamped below at 1e-3 of the largest one; the
 * edge grows by 1.25x until there are at most max(64, 4 nf) cells and at most
 * 1024 along an axis.  Memory: 12 nv + 12 nf + 4 (cells + 1) + 4 entries bytes,
 * with cells <= max(64, 4 nf) and entries = (cell, triangle) incidences.  It
 * does not depend on any voxel size.  No triangle, a face index outside
 * [0, nv) or a non-finite vertex: CG_EINVAL.  cg_mesh_info reports the grid.
 *
 * cg_voxels (registerPointCloud): the sorted unique keys of (P,3) float32 DEVICE
 * points.  It synchronises the context stream and is the call that allocates,
 * so the filter entries stay allocation-free.  P = 0 is a valid, empty set;
 * a non-finite point or res <= 0: CG_EINVAL.  cg_voxels_keys_host copies the
 * keys (K,3) int32 to the host in ascending (x, y, z) order.
 *
 * cg_filter_grasp_pose_mesh_dev: cg_filter_grasp_pose_dev with the open gripper
 * mesh tested against vox_open (the object) and the enclosed gripper mesh
 * against vox_enclosed (the background, may be NULL or empty).  Statuses,
 * offsets and poses as above, including split_coll_status; prm->sdf_mode and
 * prm->sdf_margin are ignored.  Both voxel sets must share one resolution.
 * cg_filter_grasp_pose_mesh_host: the same from HOST points; it builds the two
 * voxel sets at octo_resolution itself.                                       */
typedef struct cg_mesh cg_mesh;
typedef struct cg_voxels cg_voxels;
int  cg_mesh_create(cg_ctx *ctx, const float *V, int nv, const int32_t *F, int nf, cg_mesh **out);
void cg_mesh_destroy(cg_mesh *mesh);
int  cg_mesh_info(const cg_mesh *mesh, int dims[3], float *cell, int64_t *entries);
int  cg_voxels_create_dev(cg_ctx *ctx, const float *pts, int P, float res, cg_voxels **out);
void cg_voxels_destroy(cg_voxels *vox);
int  cg_voxels_count(const cg_voxels *vox, int *out_K);
int  cg_voxels_keys_host(cg_voxels *vox, int32_t *out_keys);
int cg_filter_grasp_pose_mesh_dev(cg_ctx *ctx, const cg_filter_params *prm,
                                  const float *grasp_poses, int G,
                                  const float *symmetry_tfs, int S,
                                  cg_mesh *mesh_open, cg_voxels *vox_open,
                                  cg_mesh *mesh_enclosed, cg_voxels *vox_enclosed,
                                  uint8_t *out_status, int8_t *out_offset, float *out_poses);
int cg_filter_grasp_pose_mesh_host(cg_ctx *ctx, const cg_filter_params *prm,
                                   const float *grasp_poses, int G,
                                   const float *symmetry_tfs, int S,
                                   cg_mesh *mesh_open, const float *open_pts, int P1,
                                   cg_mesh *mesh_enclosed, const float *enclosed_pts, int P2,
                                   float octo_resolution,
                                   uint8_t *out_status, int8_t *out_offset, float *out_poses);

/* ---- occupancy / occlusion grid from a depth scan ----------------------------
 * Replaces: my_cpp/common.cpp:324-431 (makeOccupancyGridFromCloudScan; the K
 * argument of the reference is computed with but never influences its output).
 * Samples form a regular grid over the padded bounding box of pts:
 *   dims[a] = int((max_a + 0.005 - (min_a - 0.005)) / resolution), origin[a] = min_a - 0.005   (float arithmetic)
 * out_flags[(xi*ny + yi)*nz + zi] = 1 iff the first occupied cell on the ray origin -> sample is not farther than
 * the sample (the reference pushes exactly these samples, in thread-arrival order; here raster order).            */
int cg_occupancy_grid_geometry(const float *pts_host, int P, float resolution, int dims[3], float origin[3]);
int cg_occupancy_from_scan_host(cg_ctx *ctx, const float *pts_host, int P, float resolution,
                                unsigned char *out_flags_host);

/* ---- NUNOCS 9-DoF RANSAC hypothesis scoring -------------------------------------
 * Replaces: aligning.py:36-81 (estimate9DTransform_worker) for H hypotheses at once.
 *   source, target (N,3) float64 correspondences; ids (H,4) int32 = the 4-subsets (host numpy RNG, aligning.py:91-97)
 *   out_valid[h] = hypothesis passed the scale / singular-value / det / max_dimensions gates
 *   out_ratio[h] = inlier ratio at pass_threshold, out_T[h] = (4,4) float64 transform R diag(scales) | t           */
int cg_ransac9d_host(cg_ctx *ctx, const double *source, const double *target, int N, const int32_t *ids, int H,
                     double pass_threshold, const double min_scale[3], const double max_scale[3],
                     const double *max_dims, double *out_ratio, double *out_T, unsigned char *out_valid);

/* ---- Cone pose enumeration (device pointers, float64 like the reference's numpy) ----------
 * Replaces: dexnet/grasping/grasp_sampler.py:266-286 (PointConeGraspSampler.sample_one_surface_point: the
 *   R0 / R0 @ R_sphere @ R_inplane x approach-depth loops, Utils.py:172-179 normalizeRotation) and :191-203
 *   (center_ob_between_gripper).  Its C++ twin my_cpp/common.cpp:111-153 (augmentGraspPoses) is uncalled.
 *   surface_pts (S,3), R0 (S,9 row-major: columns approach / major / minor, computed on the host, :262),
 *   R_sphere (NS,9), R_inplane (NI,9), depths (ND) = np.arange(0, hand_depth, approach_step)
 *   out_poses64 (P,16) row-major 4x4, P = S * (1 + NS*NI) * ND, ordered (surface point, rotation, depth) like the
 *   reference's list; out_poses32 (P,16) or NULL = the same poses narrowed to float32 for cg_filter_grasp_pose_dev.   */
int cg_cone_poses_dev(cg_ctx *ctx, const double *surface_pts, const double *R0, int S, const double *R_sphere, int NS,
                      const double *R_inplane, int NI, const double *depths, int ND, double init_bite,
                      double *out_poses64, float *out_poses32);
/* grasp_sampler.py:191-203: shift every pose along its y axis to the middle of the object's extent (pts (M,3) float64,
 * camera frame) in the grasp frame; poses are updated in place (poses32 may be NULL).                                */
int cg_center_grasps_dev(cg_ctx *ctx, double *poses64, float *poses32, int P, const double *pts, int M);

/* ---- Affordance transfer per grasp (device pointers, float64) --------------------------------
 * Replaces: run_grasp_simulation.py:50-73 (compute_grasp_affordance_worker) + pybullet_env/env_grasp.py:243-283
 *   (get_finger_contact_area) for G grasps at once.
 *   cam_in_finger (G,16) = inv(finger_mesh_in_grasp) * inv(grasp_in_cam) per grasp (row-major 4x4, :52)
 *   pts, nrm (P,3): the canonical cloud and normals in the camera frame; affordance (P): score of each point's nearest
 *   canonical point (:62-63, gathered once per object on the host)
 *   finger_boxes (F,4) = x min, x max, z min, z max of each finger mesh (:252); grip_dirs (F) = +1 / -1 for a finger closing
 *   along +y / -y (:261-266); 1 <= F <= 4
 *   out_p (G) = p(T|G), NaN where the reference drops the grasp; out_contacts (G,4) = contact-patch sizes per finger.   */
int cg_grasp_affordance_dev(cg_ctx *ctx, const double *cam_in_finger, int G, const double *pts, const double *nrm,
                            const double *affordance, int P, const double *finger_boxes, const int *grip_dirs, int F,
                            double surface_tol, double *out_p, int *out_contacts);

/* ---- PointNet++ primitives (device pointers) ---------------------------
 * Replace the free functions of pointnet2.py:14-149.  Indices are int32 on
 * the device (the Python mirror widens to int64 like the reference).        */
/* pointnet2.py:14-33  square_distance: (B,S,3),(B,N,3) -> (B,S,N)           */
int cg_square_distance_dev(cg_ctx *ctx, const float *src, const float *dst,
                           int B, int S, int N, float *out);
/* pointnet2.py:35-51  index_points: points (B,N,C), idx (B,S) -> (B,S,C)    */
int cg_index_points_dev(cg_ctx *ctx, const float *points, const int32_t *idx,
                        int B, int N, int C, int S, float *out);
/* pointnet2.py:54-75  farthest_point_sample with explicit start indices.
 * cg_fps_dev: one thread-block cluster per cloud, points + running distances in
 * registers, one distributed-shared-memory exchange per round (N <= 65536 /
 * 131072 points for cluster size 8 / 16).  cg_fps_single_cta_dev: the round-1
 * one-CTA kernel (N <= 56320), kept for comparison.                           */
int cg_fps_dev(cg_ctx *ctx, const float *xyz, int B, int N, int npoint,
               const int32_t *start_idx, int32_t *out_idx);
int cg_fps_single_cta_dev(cg_ctx *ctx, const float *xyz, int B, int N, int npoint,
                          const int32_t *start_idx, int32_t *out_idx);
/* pointnet2.py:78-98  query_ball_point (first nsample by index, pad w/ first;
 * an empty ball yields N in every slot, like the reference).  radius2 is
 * float32(radius**2), the threshold torch compares against (:93)            */
int cg_ball_query_dev(cg_ctx *ctx, float radius2, int nsample,
                      const float *xyz, const float *new_xyz,
                      int B, int N, int S, int32_t *out_idx);
/* pointnet2.py:101-129 grouping tail of sample_and_group:
 * out (B,S,K,3+D) = [xyz[idx]-new_xyz, points[idx]]                         */
int cg_group_points_dev(cg_ctx *ctx, const float *xyz, const float *points,
                        const float *new_xyz, const int32_t *idx,
                        int B, int N, int D, int S, int K, float *out);


/* ---- PointNet++ set-abstraction / feature-propagation stacks -----------------------------
 * The reference ships the primitives above and cites the upstream module family in its model
 * docstrings (pointnet2.py:274,304); these entry points are that family's
 * PointNetSetAbstraction / PointNetFeaturePropagation built on the primitives
 * (sample_and_group, pointnet2.py:101-129; square_distance, :14-33).
 *
 * cg_mlp: a stack of nlayers shared (1x1 conv + BatchNorm + ReLU) layers, BN folded by the host:
 *   dims[nlayers+1] channel counts, Wt_host[i] = [dims[i]][dims[i+1]] k-major fp32, b_host[i] = [dims[i+1]].
 * Layers whose input width is a multiple of 64 run on tcgen05 (bf16 hi/lo x3, fp32 accumulate) when
 * there are >= 64 rows; narrower ones (the 3+D input layer) on the FMA kernels.                        */
typedef struct cg_mlp cg_mlp;
int  cg_mlp_create(cg_ctx *ctx, int nlayers, const int *dims, const float *const *Wt_host,
                   const float *const *b_host, cg_mlp **out);
void cg_mlp_destroy(cg_mlp *mlp);
/* x (R, dims[0]) -> out (R, dims[nlayers]): the per-row MLP (feature-propagation tail).               */
int  cg_shared_mlp_dev(cg_mlp *mlp, const float *x, int64_t R, float *out);
/* grouped (G, K, dims[0]) = output of cg_group_points_dev with G = B*S -> out (G, dims[nlayers]):
 * per-row MLP over all G*K rows, then max over the K rows of every group (set abstraction).           */
int  cg_group_mlp_max_dev(cg_mlp *mlp, const float *grouped, int G, int K, float *out);
/* Feature propagation, interpolation half: for every dense point xyz1[b][n] the 3 nearest of the S
 * sparse points xyz2[b] (expanded-form distances, ties -> lower index), weights (1/(d+1e-8))/sum, and
 *   out[b][n] = [points1[b][n] (D1 skip channels, optional) | sum_j w_j * points2[b][idx_j] (D2)]
 * out (B,N,D1+D2); out_idx (B,N,3) int32 / out_weight (B,N,3) optional (NULL: scratch).  S >= 3.      */
int  cg_three_interp_dev(cg_ctx *ctx, const float *xyz1, const float *xyz2, const float *points1, int D1,
                         const float *points2, int D2, int B, int N, int S, float *out,
                         int32_t *out_idx, float *out_weight);

/* ---- point-cloud front end (device pointers, float64) ---------------------------------------
 * Replaces the open3d / scipy.spatial.cKDTree calls that turn a depth scan into the clouds of the grasp
 * stage: run_grasp_simulation.py:113-139 and :171-175 (compute_candidate_grasp_one_ob), :198-211 and
 * :245-251 (compute_candidate_grasp), Utils.py:205-213 (correct_pcd_normal_direction) and :482-488
 * (cloudA_minus_cloudB).  Distances are ((dx*dx + dy*dy) + dz*dz) in float64, no contraction.
 *
 * cg_cloud: (N,3) points plus a grid of their OCCUPIED cells (cell edge `cell`, coarse level 8*cell), memory
 * O(N).  Create copies and sorts the points and synchronises the context stream (it reads the bounding box
 * and the number of occupied cells); it is the only call that allocates.  Non-finite points or more than
 * 2^21 cells along an axis: CG_EINVAL.  N = 0 is a valid, empty cloud.                                     */
typedef struct cg_cloud cg_cloud;
int  cg_cloud_create_dev(cg_ctx *ctx, const double *pts, int N, double cell, cg_cloud **out);
void cg_cloud_destroy(cg_cloud *c);
/* cKDTree.query(q, k=1) (run_grasp_simulation.py:118-119): exact nearest point, out_dist = sqrt(d^2),
 * out_idx = its index in the create-time points; ties go to the lower index.  An empty cloud or a
 * non-finite query gives (inf, N), cKDTree's "no neighbour".                                               */
int  cg_cloud_nearest_dev(cg_cloud *c, const double *q, int Q, double *out_dist, int32_t *out_idx);
/* out[i] = 1 iff some point lies within distance <= r of q[i]: the `dists <= gripper_diameter/2` crop of
 * run_grasp_simulation.py:130-133, and cloudA_minus_cloudB (Utils.py:482-488) with the cloud = B, q = A.     */
int  cg_cloud_any_within_dev(cg_cloud *c, const double *q, int Q, double r, uint8_t *out);
/* Normals of the cloud's own points (open3d estimate_normals with KDTreeSearchParamHybrid(radius, max_nn),
 * run_grasp_simulation.py:208-210,247-249) fused with correct_pcd_normal_direction(view_port):
 * neighbours = the max_nn nearest points with d^2 < radius^2 (the point itself included, ties to the lower
 * index), covariance from the cumulants, eigenvector of its smallest eigenvalue; (0,0,1) with fewer than 3
 * neighbours; then n / (|n| + 1e-10), flipped where it points away from view_port.  1 <= max_nn <= 32.
 * out_nrm (N,3) in the create-time point order.  out_nbr (N, max_nn) int32 or NULL: the neighbour indices in
 * ascending distance, padded with N (cKDTree.query(k=max_nn, distance_upper_bound=radius) layout).          */
int  cg_cloud_normals_dev(cg_cloud *c, double radius, int max_nn, const double view_port[3], double *out_nrm,
                          int32_t *out_nbr);
/* open3d voxel_down_sample (run_grasp_simulation.py:114,137,173,246): voxel index
 * floor((p - (min - 0.5*voxel)) / voxel); every output point (and normal, if nrm != NULL) is the sum of its
 * voxel's inputs IN INPUT ORDER divided by their count (normals are not re-normalised).  Output order is
 * ascending voxel index (x, then y, then z) -- open3d emits its hash-map order, which cannot be reproduced.
 * out_pts / out_nrm need room for N rows; *out_count (DEVICE int32) receives the number of voxels.  Reads the
 * bounding box back (synchronises the stream).  voxel <= 0, non-finite input, or an index range beyond
 * int32 (open3d: "voxel_size is too small"): CG_EINVAL.                                                     */
int  cg_voxel_down_sample_dev(cg_ctx *ctx, const double *pts, const double *nrm, int N, double voxel,
                              double *out_pts, double *out_nrm, int32_t *out_count);

#ifdef __cplusplus
}
#endif
#endif /* CATGRASP_B200_H */
