// cg_pose.cuh -- pose logic of the fused grasp-pose filter (my_cpp/common.cpp:159,185-212,253-299), shared by the
// gripper-SDF predicate (cg_collide.cu) and the mesh-vs-voxel predicate (cg_mesh_collide.cu) so that both see the
// same grasp_in_cam and gripper_in_cam bit for bit.
//
// fp32 in the reference's operation order (Eigen 4x4 products without FMA contraction, column normalisation by
// division through sqrt, the float step accumulator whose 3 mm iteration never executes); every operation carries an
// explicit rounding intrinsic so that the CPU oracles can reproduce it.
#pragma once
#include "cg_common.cuh"

namespace cg_pose {

__device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }

// Eigen fixed-size 4x4 float product as compiled by the reference build (SSE2, no FMA):
// out(r,c) = ((a(r,0)b(0,c) + a(r,1)b(1,c)) + a(r,2)b(2,c)) + a(r,3)b(3,c)
__device__ inline void mm4(const float *A, const float *B, float *O) {
#pragma unroll
  for (int r = 0; r < 4; r++)
#pragma unroll
    for (int c = 0; c < 4; c++) {
      float s = mul(A[r * 4 + 0], B[0 * 4 + c]);
      s = add(s, mul(A[r * 4 + 1], B[1 * 4 + c]));
      s = add(s, mul(A[r * 4 + 2], B[2 * 4 + c]));
      s = add(s, mul(A[r * 4 + 3], B[3 * 4 + c]));
      O[r * 4 + c] = s;
    }
}

// Eigen normalize(): v /= sqrt(x*x + y*y + z*z)   (common.cpp:194-197)
__device__ inline void normalize_col(float *G, int col) {
  const float x = G[0 * 4 + col], y = G[1 * 4 + col], z = G[2 * 4 + col];
  const float n = __fsqrt_rn(add(add(mul(x, x), mul(y, y)), mul(z, z)));
  G[0 * 4 + col] = __fdiv_rn(x, n);
  G[1 * 4 + col] = __fdiv_rn(y, n);
  G[2 * 4 + col] = __fdiv_rn(z, n);
}

// inverse of the affine map A (3x3 by cofactors, fixed operation order) -> inv[12] = Rinv(9), tinv(3)
__device__ inline void affine_inverse(const float *A, float *inv) {
  const float a = A[0], b = A[1], c = A[2], d = A[4], e = A[5], f = A[6], g = A[8], h = A[9], i = A[10];
  const float c00 = sub(mul(e, i), mul(f, h));
  const float c01 = sub(mul(f, g), mul(d, i));
  const float c02 = sub(mul(d, h), mul(e, g));
  const float det = add(add(mul(a, c00), mul(b, c01)), mul(c, c02));
  const float r = __fdiv_rn(1.0f, det);
  inv[0] = mul(c00, r);
  inv[1] = mul(sub(mul(c, h), mul(b, i)), r);
  inv[2] = mul(sub(mul(b, f), mul(c, e)), r);
  inv[3] = mul(c01, r);
  inv[4] = mul(sub(mul(a, i), mul(c, g)), r);
  inv[5] = mul(sub(mul(c, d), mul(a, f)), r);
  inv[6] = mul(c02, r);
  inv[7] = mul(sub(mul(b, g), mul(a, h)), r);
  inv[8] = mul(sub(mul(a, e), mul(b, d)), r);
  const float tx = A[3], ty = A[7], tz = A[11];
#pragma unroll
  for (int k = 0; k < 3; k++)
    inv[9 + k] = -add(add(mul(inv[k * 3 + 0], tx), mul(inv[k * 3 + 1], ty)), mul(inv[k * 3 + 2], tz));
}

// grasp_in_cam of pair (pose i, symmetry j), first three columns normalised (common.cpp:159,190-197); returns true
// when the approach-direction test (:199-212) rejects it.
__device__ inline bool compose_grasp(const cg_filter_params &prm, const float *sym_j, const float *pose_i, float *g) {
  float c2c[16], tmp[16];
  mm4(prm.nocs_pose, prm.canonical_to_nocs, c2c);            // common.cpp:159
  mm4(sym_j, pose_i, tmp);                                   // :190
  mm4(c2c, tmp, g);                                          // :191
  for (int col = 0; col < 3; col++) normalize_col(g, col);   // :194-197
  if (!prm.filter_approach_dir_face_camera) return false;
  const float x = g[0], y = g[4], z = g[8];
  const float n = __fsqrt_rn(add(add(mul(x, x), mul(y, y)), mul(z, z)));
  const float zz = __fdiv_rn(z, n);
  // dot with (0,0,1): x*0 + y*0 + z*1
  const float dot = add(add(mul(__fdiv_rn(x, n), 0.f), mul(__fdiv_rn(y, n), 0.f)), mul(zz, 1.f));
  return dot < 0.f;
}

// Lateral offset k of the search (0,+),(1,+),(1,-),(2,+),(2,-) (common.cpp:253-266): cur = g shifted along its own y
// axis, gic = cur * gripper_in_grasp.  The float accumulator of :255 gives steps 0, 0.001f, 0.001f+0.001f (the 3 mm
// step never runs).
__device__ inline void offset_pose(const float *g, int k, const float *gripper_in_grasp, float *cur, float *gic) {
  const float step1 = 0.001f;
  const float step2 = __fadd_rn(step1, 0.001f);
  const float step = (k == 0) ? 0.f : ((k <= 2) ? step1 : step2);
  const float sign = (k == 0 || (k & 1)) ? 1.f : -1.f;
  for (int e = 0; e < 16; e++) cur[e] = g[e];
  for (int r = 0; r < 3; r++)                                // :265  t += (step*major_dir)*sign
    cur[r * 4 + 3] = add(cur[r * 4 + 3], mul(mul(step, g[r * 4 + 1]), sign));
  mm4(cur, gripper_in_grasp, gic);                           // :266
}

}  // namespace cg_pose
