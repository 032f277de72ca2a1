// cg_mesh_collide.cu -- the reference's own geometry predicate for the grasp-pose filter: the posed gripper MESH
// touches an OCCUPIED OCTREE VOXEL (my_cpp/collision_manager.cpp:15-111, FCL BVH x octomap OcTree), without any SDF.
//
//   cg_mesh    registerMesh: the gripper-frame triangles plus a uniform grid with per-cell triangle lists (CSR).
//   cg_voxels  registerPointCloud: the sorted unique octomap keys floor(double(x) * (1.0 / res)) of a point set.
//   filter     the pose logic of cg_collide.cu (shared through cg_pose.cuh), with "collides" decided per occupied
//              cube by a gripper-frame broad phase and an exact float64 13-axis separating-axis test against the
//              posed triangles (the semantic of oracle/mesh_voxel_ref.py, bit for bit).
#include <cub/cub.cuh>

#include <algorithm>
#include <cmath>

#include "cg_common.cuh"
#include "cg_pose.cuh"

struct cg_mesh {
  cg_ctx *ctx;
  float *V = nullptr;         // device (nv,3), gripper frame
  int32_t *F = nullptr;       // device (nf,3)
  int32_t *start = nullptr;   // device (ncells+1): CSR offsets of the per-cell triangle lists
  int32_t *tris = nullptr;    // device: triangle ids, cell after cell
  int nv = 0, nf = 0;
  int dims[3];
  float org[3], cell;         // cell (x,y,z) spans org + cell * [x, x+1] (closed) per axis
  float lo[3], hi[3];         // bounding box of the vertices
  long entries = 0;
};

struct cg_voxels {
  cg_ctx *ctx;
  unsigned long long *keys = nullptr;   // device, ascending; (x+32768) << 32 | (y+32768) << 16 | (z+32768)
  int K = 0;
  double res = 0.0;                     // double(float32 resolution)
};

namespace {

using namespace cg_pose;

constexpr int KEY_LIMIT = 32768;                          // octomap: 16-bit keys, tree_max_val
constexpr unsigned long long KEY_DROPPED = 1ull << 48;    // sorts after every valid key
constexpr int MAX_AXIS_CELLS = 1024;                      // queue entries pack a cell index in 10 bits per axis

// ---------------------------------------------------------------------------- registerPointCloud
__global__ void voxel_key_kernel(const float *__restrict__ pts, int P, double inv_res, unsigned long long *__restrict__ keys,
                                 int *__restrict__ counters) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  unsigned long long key = 0;
  bool ok = true;
#pragma unroll
  for (int a = 0; a < 3; a++) {
    const double x = (double)pts[3 * (size_t)p + a];
    if (!isfinite(x)) { atomicAdd(&counters[0], 1); ok = false; break; }
    const double k = floor(__dmul_rn(x, inv_res));   // octomap coordToKey: floor(resolution_factor * coordinate)
    if (!(k >= -(double)KEY_LIMIT && k < (double)KEY_LIMIT)) { ok = false; continue; }
    key = (key << 16) | (unsigned long long)((int)k + KEY_LIMIT);
  }
  if (!ok) atomicAdd(&counters[1], 1);
  keys[p] = ok ? key : KEY_DROPPED;
}

// ---------------------------------------------------------------------------- predicate
struct MeshView {
  const float *V;
  const int32_t *F, *start, *tris;
  int nx, ny, nz;
  float ox, oy, oz, inv_cell;
  float lx, ly, lz, hx, hy, hz;
};

struct VoxView {
  const unsigned long long *keys;
  int K;
  double res;
};

struct PoseS {            // per (pair, offset), written by thread 0
  double T[12];           // gripper_in_cam rows 0..2, widened from float32
  float A[12];            // its affine inverse (float32): camera -> gripper frame, broad phase only
  float ext[3];           // gripper-frame half extent of a voxel cube, plus slack
};

__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }

__device__ __forceinline__ void key_centre(unsigned long long k, double res, double *c) {
  c[0] = dmul((double)((int)((k >> 32) & 0xffff) - KEY_LIMIT) + 0.5, res);
  c[1] = dmul((double)((int)((k >> 16) & 0xffff) - KEY_LIMIT) + 0.5, res);
  c[2] = dmul((double)((int)(k & 0xffff) - KEY_LIMIT) + 0.5, res);
}

// one SAT axis: projections (dx*ax + dy*ay) + dz*az of the three vertex offsets against half*((|ax|+|ay|)+|az|)
__device__ __forceinline__ bool axis_separates(const double d[3][3], double ax, double ay, double az, double half) {
  double p[3];
#pragma unroll
  for (int i = 0; i < 3; i++) p[i] = dadd(dadd(dmul(d[i][0], ax), dmul(d[i][1], ay)), dmul(d[i][2], az));
  const double r = dmul(half, dadd(dadd(fabs(ax), fabs(ay)), fabs(az)));
  const double lo = fmin(fmin(p[0], p[1]), p[2]), hi = fmax(fmax(p[0], p[1]), p[2]);
  return lo > r || hi < -r;
}

// Cube (centre c, half side) vs posed triangle v: true iff no axis separates (touching counts as overlap).
__device__ bool tri_cube_overlap(const double v[3][3], const double *c, double half) {
  double d[3][3];
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int a = 0; a < 3; a++) d[i][a] = dsub(v[i][a], c[a]);
#pragma unroll
  for (int a = 0; a < 3; a++) {
    const double lo = fmin(fmin(d[0][a], d[1][a]), d[2][a]), hi = fmax(fmax(d[0][a], d[1][a]), d[2][a]);
    if (lo > half || hi < -half) return false;
  }
  double e[3][3];
#pragma unroll
  for (int a = 0; a < 3; a++) {
    e[0][a] = dsub(v[1][a], v[0][a]);
    e[1][a] = dsub(v[2][a], v[1][a]);
    e[2][a] = dsub(v[0][a], v[2][a]);
  }
  if (axis_separates(d, dsub(dmul(e[0][1], e[1][2]), dmul(e[0][2], e[1][1])),
                     dsub(dmul(e[0][2], e[1][0]), dmul(e[0][0], e[1][2])),
                     dsub(dmul(e[0][0], e[1][1]), dmul(e[0][1], e[1][0])), half))
    return false;
  // cross(eye[a], e_k): (0,-ez,ey), (ez,0,-ex), (-ey,ex,0); the zero components add exactly +-0 to a projection
#pragma unroll
  for (int k = 0; k < 3; k++) {
    if (axis_separates(d, 0.0, -e[k][2], e[k][1], half)) return false;
    if (axis_separates(d, e[k][2], 0.0, -e[k][0], half)) return false;
    if (axis_separates(d, -e[k][1], e[k][0], 0.0, half)) return false;
  }
  return true;
}

// Vc = ((R0*vx + R1*vy) + R2*vz) + t, float64, no contraction
__device__ __forceinline__ void pose_vertex(const double *T, const float *__restrict__ V, int idx, double *out) {
  const double x = (double)__ldg(V + 3 * (size_t)idx), y = (double)__ldg(V + 3 * (size_t)idx + 1),
               z = (double)__ldg(V + 3 * (size_t)idx + 2);
#pragma unroll
  for (int r = 0; r < 3; r++) out[r] = dadd(dadd(dadd(dmul(T[r * 4 + 0], x), dmul(T[r * 4 + 1], y)), dmul(T[r * 4 + 2], z)), T[r * 4 + 3]);
}

constexpr int FT = 256;
constexpr int NW = FT / 32;

// Voxels that survive the broad phase are queued (key index + covered cell box) so that the float64 narrow phase runs
// one warp per voxel with the lanes over its triangle lists, whatever the broad-phase outcome of the neighbours.
constexpr int QCAP = 4 * FT;
struct VoxQueue {
  int idx[QCAP];
  unsigned lo[QCAP], hi[QCAP];   // cell box, 10 bits per axis
  int count[2];
};

__device__ __forceinline__ unsigned pack3(int x, int y, int z) { return ((unsigned)x << 20) | ((unsigned)y << 10) | (unsigned)z; }

__device__ __forceinline__ int cell_index(float x, float org, float inv_cell, int n) {
  return min(n - 1, max(0, (int)floorf((x - org) * inv_cell)));
}

// Broad phase of one voxel: gripper-frame bounding box of the cube -> covered cells; false when it misses the mesh box
// or every covered cell is empty.
__device__ __forceinline__ bool broad_phase(const MeshView &m, const PoseS &ps, double res, unsigned long long key,
                                            unsigned *clo, unsigned *chi) {
  double c[3];
  key_centre(key, res, c);
  const float fx = (float)c[0], fy = (float)c[1], fz = (float)c[2];
  const float *A = ps.A;
  const float ux = fmaf(A[2], fz, fmaf(A[1], fy, fmaf(A[0], fx, A[9])));
  const float uy = fmaf(A[5], fz, fmaf(A[4], fy, fmaf(A[3], fx, A[10])));
  const float uz = fmaf(A[8], fz, fmaf(A[7], fy, fmaf(A[6], fx, A[11])));
  const float ax = ux - ps.ext[0], bx = ux + ps.ext[0];
  const float ay = uy - ps.ext[1], by = uy + ps.ext[1];
  const float az = uz - ps.ext[2], bz = uz + ps.ext[2];
  if (bx < m.lx || ax > m.hx || by < m.ly || ay > m.hy || bz < m.lz || az > m.hz) return false;
  // both ends clamped into the grid: the box overlaps the mesh box, so the clamped range is never empty
  const int x0 = cell_index(ax, m.ox, m.inv_cell, m.nx), x1 = cell_index(bx, m.ox, m.inv_cell, m.nx);
  const int y0 = cell_index(ay, m.oy, m.inv_cell, m.ny), y1 = cell_index(by, m.oy, m.inv_cell, m.ny);
  const int z0 = cell_index(az, m.oz, m.inv_cell, m.nz), z1 = cell_index(bz, m.oz, m.inv_cell, m.nz);
  int n = 0;
  for (int x = x0; x <= x1; x++)
    for (int y = y0; y <= y1; y++) {
      const int base = (x * m.ny + y) * m.nz;
      n += __ldg(m.start + base + z1 + 1) - __ldg(m.start + base + z0);   // a z-run of cells is contiguous in the CSR
    }
  *clo = pack3(x0, y0, z0);
  *chi = pack3(x1, y1, z1);
  return n > 0;
}

// Narrow phase of one queued voxel by one warp: true (on every lane) iff some listed triangle overlaps the cube.
__device__ bool warp_narrow(const MeshView &m, const PoseS &ps, double res, unsigned long long key, unsigned clo,
                            unsigned chi) {
  const int lane = threadIdx.x & 31;
  double c[3];
  key_centre(key, res, c);
  const double half = dmul(0.5, res);
  const int x0 = clo >> 20, y0 = (clo >> 10) & 1023, z0 = clo & 1023;
  const int x1 = chi >> 20, y1 = (chi >> 10) & 1023, z1 = chi & 1023;
  for (int x = x0; x <= x1; x++)
    for (int y = y0; y <= y1; y++) {
      const int base = (x * m.ny + y) * m.nz;
      const int s = __ldg(m.start + base + z0), e = __ldg(m.start + base + z1 + 1);
      bool hit = false;
      for (int t = s + lane; t < e && !hit; t += 32) {
        const int f = __ldg(m.tris + t);
        double v[3][3];
#pragma unroll
        for (int i = 0; i < 3; i++) pose_vertex(ps.T, m.V, __ldg(m.F + 3 * (size_t)f + i), v[i]);
        hit = tri_cube_overlap(v, c, half);
      }
      if (__any_sync(0xffffffffu, hit)) return true;
    }
  return false;
}

// Scans voxels keys[0], keys[stride], ..., keys[(n-1)*stride].
__device__ bool any_voxel_hits(const MeshView &m, const PoseS &ps, const VoxView &vx, int n, int stride, VoxQueue &Q) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned lt = (1u << lane) - 1u;
  int cur = 0;
  if (threadIdx.x == 0) { Q.count[0] = 0; Q.count[1] = 0; }
  __syncthreads();
  for (int base = 0; base < n; base += 4 * FT) {
    unsigned long long k[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int p = base + j * FT + threadIdx.x;
      k[j] = p < n ? __ldg(vx.keys + (size_t)p * stride) : 0ull;
    }
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int p = base + j * FT + threadIdx.x;
      unsigned clo = 0, chi = 0;
      const bool need = p < n && broad_phase(m, ps, vx.res, k[j], &clo, &chi);
      const unsigned msk = __ballot_sync(0xffffffffu, need);
      if (msk) {
        int at = 0;
        if (lane == 0) at = atomicAdd(&Q.count[cur], __popc(msk));
        at = __shfl_sync(0xffffffffu, at, 0);
        if (need) {
          const int e = at + __popc(msk & lt);
          Q.idx[e] = p; Q.lo[e] = clo; Q.hi[e] = chi;
        }
      }
    }
    __syncthreads();
    const int nq = Q.count[cur];
    if (threadIdx.x == 0) Q.count[cur ^ 1] = 0;      // next chunk's counter; nobody touches it before the barrier below
    bool hit = false;
    for (int e = warp; e < nq && !hit; e += NW)
      hit = warp_narrow(m, ps, vx.res, __ldg(vx.keys + (size_t)Q.idx[e] * stride), Q.lo[e], Q.hi[e]);
    if (__syncthreads_or(hit)) return true;
    cur ^= 1;
  }
  return false;
}

// thread 0: the per-offset pose data of the predicate
__device__ void pose_setup(const float *gic, PoseS &ps, double res) {
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 4; c++) ps.T[r * 4 + c] = (double)gic[r * 4 + c];
  affine_inverse(gic, ps.A);
  // slack over the float32 rounding of the centre, the inverse and the transform (each a few ulp of |t| ~ 1 m):
  // 1e-5 m plus 1e-5 of the translation's and the inverse's magnitude, orders of magnitude above that
  const float tmax = fmaxf(fmaxf(fabsf(gic[3]), fabsf(gic[7])), fabsf(gic[11]));
  const float h = (float)(0.5 * res);
  for (int r = 0; r < 3; r++) {
    const float s = fabsf(ps.A[r * 3 + 0]) + fabsf(ps.A[r * 3 + 1]) + fabsf(ps.A[r * 3 + 2]);
    ps.ext[r] = h * s * 1.0001f + 1e-5f * (1.f + tmax * s);
  }
}

__global__ void __launch_bounds__(FT) mesh_filter_kernel(const cg_filter_params prm, const float *__restrict__ grasp_poses,
                                                         int G, const float *__restrict__ sym, int S, MeshView mesh_open,
                                                         VoxView vox_open, MeshView mesh_encl, VoxView vox_encl,
                                                         uint8_t *__restrict__ out_status, int8_t *__restrict__ out_offset,
                                                         float *__restrict__ out_poses) {
  __shared__ float g_s[16];      // grasp_in_cam (normalised)
  __shared__ float cur_s[16];    // shifted candidate
  __shared__ PoseS ps;
  __shared__ int rej_dir;
  __shared__ VoxQueue vq;
  const long q = blockIdx.x;
  const int i = (int)(q / S), j = (int)(q % S);
  if (threadIdx.x == 0) {
    float g[16];
    rej_dir = compose_grasp(prm, sym + (size_t)j * 16, grasp_poses + (size_t)i * 16, g);
    for (int k = 0; k < 16; k++) g_s[k] = g[k];
  }
  __syncthreads();
  if (rej_dir) {
    if (threadIdx.x == 0) { out_status[q] = CG_ST_REJ_DIR; out_offset[q] = -1; }
    if (threadIdx.x < 16) out_poses[q * 16 + threadIdx.x] = 0.f;
    return;
  }
  const int n_off = prm.adjust_collision_pose ? 5 : 1;
  const bool split = prm.split_coll_status && !prm.adjust_collision_pose;
  const int P1 = vox_open.K, P2 = vox_encl.K;
  bool open_hit = false;
  int winner = -1;
  for (int k = 0; k < n_off; k++) {
    if (threadIdx.x == 0) {
      float cur[16], gic[16];
      offset_pose(g_s, k, prm.gripper_in_grasp, cur, gic);
      pose_setup(gic, ps, vox_open.res);
      for (int e = 0; e < 16; e++) cur_s[e] = cur[e];
    }
    __syncthreads();
    // same scan order as the SDF filter (cg_collide.cu): a strided sample of the background voxels, the object's,
    // then every background voxel; split status keeps the reference's order (open gripper first)
    const int head = min(P2, 4 * FT);
    const int hstride = head > 0 ? P2 / head : 1;
    bool coll;
    if (split) {
      coll = any_voxel_hits(mesh_open, ps, vox_open, P1, 1, vq);
      open_hit = coll;
      if (!coll && head > 0) coll = any_voxel_hits(mesh_encl, ps, vox_encl, head, hstride, vq);
    } else {
      coll = (head > 0) && any_voxel_hits(mesh_encl, ps, vox_encl, head, hstride, vq);
      if (!coll) coll = any_voxel_hits(mesh_open, ps, vox_open, P1, 1, vq);
    }
    if (!coll && P2 > head) coll = any_voxel_hits(mesh_encl, ps, vox_encl, P2, 1, vq);
    if (!coll) { winner = k; break; }
    __syncthreads();  // everyone is done reading ps before thread 0 rewrites it
  }
  if (threadIdx.x == 0) {
    out_status[q] = (winner >= 0) ? CG_ST_ACCEPT : ((split && !open_hit) ? CG_ST_REJ_COLL_ENCL : CG_ST_REJ_COLL);
    out_offset[q] = (int8_t)winner;
  }
  if (threadIdx.x < 16) out_poses[q * 16 + threadIdx.x] = (winner >= 0) ? cur_s[threadIdx.x] : 0.f;
}

MeshView view(const cg_mesh *m) {
  MeshView v;
  v.V = m->V; v.F = m->F; v.start = m->start; v.tris = m->tris;
  v.nx = m->dims[0]; v.ny = m->dims[1]; v.nz = m->dims[2];
  v.ox = m->org[0]; v.oy = m->org[1]; v.oz = m->org[2];
  v.inv_cell = 1.0f / m->cell;
  v.lx = m->lo[0]; v.ly = m->lo[1]; v.lz = m->lo[2];
  v.hx = m->hi[0]; v.hy = m->hi[1]; v.hz = m->hi[2];
  return v;
}

VoxView view(const cg_voxels *v) { return VoxView{v->keys, v->K, v->res}; }

// ---------------------------------------------------------------------------- registerMesh (host)
// Conservative triangle vs closed box (centre c, half extent h) in double: the 13-axis SAT.
bool host_tri_box(const double v[3][3], const double c[3], double h) {
  double d[3][3], e[3][3];
  for (int i = 0; i < 3; i++)
    for (int a = 0; a < 3; a++) d[i][a] = v[i][a] - c[a];
  for (int a = 0; a < 3; a++) {
    e[0][a] = v[1][a] - v[0][a]; e[1][a] = v[2][a] - v[1][a]; e[2][a] = v[0][a] - v[2][a];
  }
  auto sep = [&](double ax, double ay, double az) {
    double lo = 1e300, hi = -1e300;
    for (int i = 0; i < 3; i++) {
      const double p = d[i][0] * ax + d[i][1] * ay + d[i][2] * az;
      lo = std::min(lo, p); hi = std::max(hi, p);
    }
    const double r = h * (std::fabs(ax) + std::fabs(ay) + std::fabs(az));
    return lo > r || hi < -r;
  };
  if (sep(1, 0, 0) || sep(0, 1, 0) || sep(0, 0, 1)) return false;
  if (sep(e[0][1] * e[1][2] - e[0][2] * e[1][1], e[0][2] * e[1][0] - e[0][0] * e[1][2], e[0][0] * e[1][1] - e[0][1] * e[1][0]))
    return false;
  for (int k = 0; k < 3; k++)
    if (sep(0, -e[k][2], e[k][1]) || sep(e[k][2], 0, -e[k][0]) || sep(-e[k][1], e[k][0], 0)) return false;
  return true;
}

inline unsigned blocks(long n, int t) { return (unsigned)((n + t - 1) / t); }

}  // namespace

extern "C" int cg_mesh_create(cg_ctx *ctx, const float *V, int nv, const int32_t *F, int nf, cg_mesh **out) {
  if (!ctx || !out) return CG_EINVAL;
  *out = nullptr;
  CG_REQUIRE(ctx, V && F && nv > 0 && nf > 0, "mesh_create: need vertices and at least one triangle");
  for (long i = 0; i < 3L * nv; i++) CG_REQUIRE(ctx, std::isfinite(V[i]), "mesh_create: non-finite vertex");
  for (long i = 0; i < 3L * nf; i++) CG_REQUIRE(ctx, F[i] >= 0 && F[i] < nv, "mesh_create: face index out of range");
  float lo[3], hi[3];
  for (int a = 0; a < 3; a++) { lo[a] = V[a]; hi[a] = V[a]; }
  for (int i = 1; i < nv; i++)
    for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], V[3 * i + a]); hi[a] = std::max(hi[a], V[3 * i + a]); }
  // Cell-size rule: cubic cells, about 2 cells per triangle over the bounding box, at most max(64, 4 nf) cells and
  // MAX_AXIS_CELLS per axis (each axis gets floor(extent / cell) + 1 cells).
  double ext[3], emax = 0.0;
  for (int a = 0; a < 3; a++) { ext[a] = (double)hi[a] - (double)lo[a]; emax = std::max(emax, ext[a]); }
  if (emax <= 0.0) emax = 1e-6;
  double vol = 1.0;
  for (int a = 0; a < 3; a++) vol *= std::max(ext[a], 1e-3 * emax);
  double cell = std::max(std::cbrt(vol / (2.0 * nf)), emax / (MAX_AXIS_CELLS - 1));
  int dims[3];
  const long cap = std::max(64L, 4L * nf);
  for (;;) {
    const float cf = (float)cell;
    long n = 1;
    for (int a = 0; a < 3; a++) { dims[a] = (int)std::floor(ext[a] / cf) + 1; n *= dims[a]; }
    if (n <= cap && dims[0] <= MAX_AXIS_CELLS && dims[1] <= MAX_AXIS_CELLS && dims[2] <= MAX_AXIS_CELLS) break;
    cell *= 1.25;
  }
  const float cf = (float)cell;
  const long ncells = (long)dims[0] * dims[1] * dims[2];
  // Per-cell lists: every triangle that meets the closed cell, enlarged by 1e-3 cell on each side so that the
  // kernel's float32 cell indexing can never skip a listed cell.
  std::vector<int32_t> count(ncells + 1, 0);
  std::vector<std::pair<int32_t, int32_t>> pairs;   // (cell, triangle)
  const double h = 0.5 * cf * (1.0 + 2e-3);
  for (int t = 0; t < nf; t++) {
    double v[3][3];
    int c0[3], c1[3];
    for (int i = 0; i < 3; i++)
      for (int a = 0; a < 3; a++) v[i][a] = (double)V[3 * F[3 * t + i] + a];
    for (int a = 0; a < 3; a++) {
      const double mn = std::min(v[0][a], std::min(v[1][a], v[2][a])), mx = std::max(v[0][a], std::max(v[1][a], v[2][a]));
      c0[a] = std::max(0, (int)std::floor((mn - lo[a]) / cf - 1e-3));
      c1[a] = std::min(dims[a] - 1, (int)std::floor((mx - lo[a]) / cf + 1e-3));
    }
    for (int x = c0[0]; x <= c1[0]; x++)
      for (int y = c0[1]; y <= c1[1]; y++)
        for (int z = c0[2]; z <= c1[2]; z++) {
          const double c[3] = {lo[0] + (x + 0.5) * (double)cf, lo[1] + (y + 0.5) * (double)cf, lo[2] + (z + 0.5) * (double)cf};
          if (!host_tri_box(v, c, h)) continue;
          const int32_t lin = (int32_t)(((long)x * dims[1] + y) * dims[2] + z);
          pairs.emplace_back(lin, t);
          count[lin + 1]++;
        }
  }
  CG_REQUIRE(ctx, pairs.size() < (size_t)INT32_MAX, "mesh_create: too many cell entries");
  for (long c = 0; c < ncells; c++) count[c + 1] += count[c];
  std::vector<int32_t> tris(pairs.size());
  {
    std::vector<int32_t> fill(count.begin(), count.end() - 1);
    for (const auto &p : pairs) tris[fill[p.first]++] = p.second;   // triangles ascending within a cell
  }
  CG_CUDA(ctx, cudaSetDevice(ctx->device));
  cg_mesh *m = new cg_mesh();
  m->ctx = ctx; m->nv = nv; m->nf = nf; m->cell = cf; m->entries = (long)tris.size();
  for (int a = 0; a < 3; a++) { m->dims[a] = dims[a]; m->org[a] = lo[a]; m->lo[a] = lo[a]; m->hi[a] = hi[a]; }
  auto fail = [&](cudaError_t e) {
    ctx->err = std::string("mesh_create: ") + cudaGetErrorString(e);
    cudaFree(m->V); cudaFree(m->F); cudaFree(m->start); cudaFree(m->tris);
    delete m;
    return CG_ECUDA;
  };
  cudaError_t e;
  if ((e = cudaMalloc(&m->V, (size_t)nv * 12)) != cudaSuccess) return fail(e);
  if ((e = cudaMalloc(&m->F, (size_t)nf * 12)) != cudaSuccess) return fail(e);
  if ((e = cudaMalloc(&m->start, (size_t)(ncells + 1) * 4)) != cudaSuccess) return fail(e);
  if ((e = cudaMalloc(&m->tris, std::max<size_t>(tris.size(), 1) * 4)) != cudaSuccess) return fail(e);
  if ((e = cudaMemcpy(m->V, V, (size_t)nv * 12, cudaMemcpyHostToDevice)) != cudaSuccess) return fail(e);
  if ((e = cudaMemcpy(m->F, F, (size_t)nf * 12, cudaMemcpyHostToDevice)) != cudaSuccess) return fail(e);
  if ((e = cudaMemcpy(m->start, count.data(), (size_t)(ncells + 1) * 4, cudaMemcpyHostToDevice)) != cudaSuccess) return fail(e);
  if (!tris.empty() && (e = cudaMemcpy(m->tris, tris.data(), tris.size() * 4, cudaMemcpyHostToDevice)) != cudaSuccess)
    return fail(e);
  *out = m;
  return CG_OK;
}

extern "C" void cg_mesh_destroy(cg_mesh *m) {
  if (!m) return;
  cudaSetDevice(m->ctx->device);
  cudaFree(m->V); cudaFree(m->F); cudaFree(m->start); cudaFree(m->tris);
  delete m;
}

extern "C" int cg_mesh_info(const cg_mesh *m, int dims[3], float *cell, int64_t *entries) {
  if (!m || !dims || !cell || !entries) return CG_EINVAL;
  for (int a = 0; a < 3; a++) dims[a] = m->dims[a];
  *cell = m->cell;
  *entries = m->entries;
  return CG_OK;
}

extern "C" int cg_voxels_create_dev(cg_ctx *ctx, const float *pts, int P, float res, cg_voxels **out) {
  if (!ctx || !out) return CG_EINVAL;
  *out = nullptr;
  CG_REQUIRE(ctx, P >= 0 && (pts || P == 0), "voxels_create: bad points");
  CG_REQUIRE(ctx, res > 0.f && std::isfinite(res), "voxels_create: resolution must be positive and finite");
  CG_CUDA(ctx, cudaSetDevice(ctx->device));
  const double r = (double)res;
  if (P == 0) {
    cg_voxels *v = new cg_voxels();
    v->ctx = ctx; v->res = r;
    *out = v;
    return CG_OK;
  }
  size_t sort_b = 0, uniq_b = 0;
  cub::DeviceRadixSort::SortKeys(nullptr, sort_b, (unsigned long long *)nullptr, (unsigned long long *)nullptr, P, 0, 49);
  cub::DeviceSelect::Unique(nullptr, uniq_b, (unsigned long long *)nullptr, (unsigned long long *)nullptr, (int *)nullptr, P);
  const size_t cub_b = std::max(sort_b, uniq_b);
  const size_t ws = 3 * cg_arena::pad((size_t)P * 8) + cg_arena::pad(4 * sizeof(int)) + cg_arena::pad(cub_b);
  int rc = cg_ws_reserve(ctx, ws);
  if (rc) return rc;
  cg_arena ar(ctx->ws);
  auto *k0 = ar.take<unsigned long long>(P), *k1 = ar.take<unsigned long long>(P), *uq = ar.take<unsigned long long>(P);
  int *cnt = ar.take<int>(4);
  void *tmp = ar.take<char>(cub_b);
  cudaStream_t st = ctx->stream;
  CG_CUDA(ctx, cudaMemsetAsync(cnt, 0, 4 * sizeof(int), st));
  voxel_key_kernel<<<blocks(P, 256), 256, 0, st>>>(pts, P, 1.0 / r, k0, cnt);   // octomap: resolution_factor = 1.0 / res
  CG_LAUNCH_CHECK(ctx);
  size_t b = cub_b;
  CG_CUDA(ctx, cub::DeviceRadixSort::SortKeys(tmp, b, k0, k1, P, 0, 49, st));
  b = cub_b;
  CG_CUDA(ctx, cub::DeviceSelect::Unique(tmp, b, k1, uq, cnt + 2, P, st));
  int h[4];
  CG_CUDA(ctx, cudaMemcpyAsync(h, cnt, sizeof(h), cudaMemcpyDeviceToHost, st));
  CG_CUDA(ctx, cudaStreamSynchronize(st));
  CG_REQUIRE(ctx, h[0] == 0, "voxels_create: point coordinates must be finite");
  const int K = h[2] - (h[1] > 0 ? 1 : 0);   // the dropped-point marker is one run at the end
  cg_voxels *v = new cg_voxels();
  v->ctx = ctx; v->res = r; v->K = K;
  if (K > 0) {
    cudaError_t e = cudaMalloc(&v->keys, (size_t)K * 8);
    if (e == cudaSuccess) e = cudaMemcpyAsync(v->keys, uq, (size_t)K * 8, cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
      ctx->err = std::string("voxels_create: ") + cudaGetErrorString(e);
      cudaFree(v->keys);
      delete v;
      return CG_ECUDA;
    }
  }
  *out = v;
  return CG_OK;
}

extern "C" void cg_voxels_destroy(cg_voxels *v) {
  if (!v) return;
  cudaSetDevice(v->ctx->device);
  cudaFree(v->keys);
  delete v;
}

extern "C" int cg_voxels_count(const cg_voxels *v, int *out_K) {
  if (!v || !out_K) return CG_EINVAL;
  *out_K = v->K;
  return CG_OK;
}

extern "C" int cg_voxels_keys_host(cg_voxels *v, int32_t *out_keys) {
  if (!v) return CG_EINVAL;
  cg_ctx *ctx = v->ctx;
  CG_REQUIRE(ctx, out_keys || v->K == 0, "voxels_keys: null output");
  if (v->K == 0) return CG_OK;
  CG_CUDA(ctx, cudaSetDevice(ctx->device));
  std::vector<unsigned long long> k(v->K);
  CG_CUDA(ctx, cudaMemcpyAsync(k.data(), v->keys, (size_t)v->K * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < v->K; i++) {
    out_keys[3 * i + 0] = (int32_t)((k[i] >> 32) & 0xffff) - KEY_LIMIT;
    out_keys[3 * i + 1] = (int32_t)((k[i] >> 16) & 0xffff) - KEY_LIMIT;
    out_keys[3 * i + 2] = (int32_t)(k[i] & 0xffff) - KEY_LIMIT;
  }
  return CG_OK;
}

extern "C" int cg_filter_grasp_pose_mesh_dev(cg_ctx *ctx, const cg_filter_params *prm, const float *grasp_poses, int G,
                                             const float *symmetry_tfs, int S, cg_mesh *mesh_open, cg_voxels *vox_open,
                                             cg_mesh *mesh_enclosed, cg_voxels *vox_enclosed, uint8_t *out_status,
                                             int8_t *out_offset, float *out_poses) {
  if (!ctx) return CG_EINVAL;
  CG_REQUIRE(ctx, prm && grasp_poses && symmetry_tfs && G > 0 && S > 0, "mesh filter: poses");
  CG_REQUIRE(ctx, mesh_open && vox_open, "mesh filter: open gripper mesh / voxels");
  CG_REQUIRE(ctx, !vox_enclosed || vox_enclosed->K == 0 || mesh_enclosed, "mesh filter: enclosed gripper mesh");
  CG_REQUIRE(ctx, !vox_enclosed || vox_enclosed->res == vox_open->res, "mesh filter: both voxel sets need one resolution");
  CG_REQUIRE(ctx, mesh_open->ctx == ctx && vox_open->ctx == ctx, "mesh filter: handles of another context");
  CG_REQUIRE(ctx, out_status && out_offset && out_poses, "mesh filter: outputs");
  CG_REQUIRE(ctx, (long)G * S < 2147483647L, "mesh filter: too many pairs");
  CG_CUDA(ctx, cudaSetDevice(ctx->device));
  const MeshView mo = view(mesh_open);
  const MeshView me = mesh_enclosed ? view(mesh_enclosed) : mo;
  const VoxView vo = view(vox_open);
  const VoxView ve = vox_enclosed ? view(vox_enclosed) : VoxView{nullptr, 0, vox_open->res};
  mesh_filter_kernel<<<(unsigned)((long)G * S), FT, 0, ctx->stream>>>(*prm, grasp_poses, G, symmetry_tfs, S, mo, vo, me, ve,
                                                                      out_status, out_offset, out_poses);
  CG_LAUNCH_CHECK(ctx);
  return CG_OK;
}

extern "C" int cg_filter_grasp_pose_mesh_host(cg_ctx *ctx, const cg_filter_params *prm, const float *grasp_poses, int G,
                                              const float *symmetry_tfs, int S, cg_mesh *mesh_open, const float *open_pts,
                                              int P1, cg_mesh *mesh_enclosed, const float *enclosed_pts, int P2,
                                              float octo_resolution, uint8_t *out_status, int8_t *out_offset,
                                              float *out_poses) {
  if (!ctx) return CG_EINVAL;
  CG_REQUIRE(ctx, prm && grasp_poses && symmetry_tfs && G > 0 && S > 0, "mesh filter_host: poses");
  CG_REQUIRE(ctx, P1 >= 0 && P2 >= 0 && (P1 == 0 || open_pts) && (P2 == 0 || enclosed_pts), "mesh filter_host: points");
  CG_REQUIRE(ctx, out_status && out_offset && out_poses, "mesh filter_host: outputs");
  CG_REQUIRE(ctx, (long)G * S < 2147483647L, "mesh filter_host: too many pairs");
  CG_CUDA(ctx, cudaSetDevice(ctx->device));
  const size_t Q = (size_t)G * S;
  const size_t need = cg_arena::pad((size_t)G * 64) + cg_arena::pad((size_t)S * 64) + cg_arena::pad((size_t)P1 * 12 + 4) +
                      cg_arena::pad((size_t)P2 * 12 + 4) + cg_arena::pad(Q) * 2 + cg_arena::pad(Q * 64) + 4096;
  int rc = cg_io_reserve(ctx, need);
  if (rc) return rc;
  cg_arena ar(ctx->io);
  float *d_g = ar.take<float>((size_t)G * 16);
  float *d_s = ar.take<float>((size_t)S * 16);
  float *d_p1 = ar.take<float>((size_t)P1 * 3 + 1);
  float *d_p2 = ar.take<float>((size_t)P2 * 3 + 1);
  uint8_t *d_st = ar.take<uint8_t>(Q);
  int8_t *d_of = ar.take<int8_t>(Q);
  float *d_po = ar.take<float>(Q * 16);
  cudaStream_t st = ctx->stream;
  CG_CUDA(ctx, cudaMemcpyAsync(d_g, grasp_poses, (size_t)G * 64, cudaMemcpyHostToDevice, st));
  CG_CUDA(ctx, cudaMemcpyAsync(d_s, symmetry_tfs, (size_t)S * 64, cudaMemcpyHostToDevice, st));
  if (P1 > 0) CG_CUDA(ctx, cudaMemcpyAsync(d_p1, open_pts, (size_t)P1 * 12, cudaMemcpyHostToDevice, st));
  if (P2 > 0) CG_CUDA(ctx, cudaMemcpyAsync(d_p2, enclosed_pts, (size_t)P2 * 12, cudaMemcpyHostToDevice, st));
  cg_voxels *vo = nullptr, *ve = nullptr;
  rc = cg_voxels_create_dev(ctx, d_p1, P1, octo_resolution, &vo);
  if (!rc) rc = cg_voxels_create_dev(ctx, d_p2, P2, octo_resolution, &ve);
  if (!rc) rc = cg_filter_grasp_pose_mesh_dev(ctx, prm, d_g, G, d_s, S, mesh_open, vo, mesh_enclosed, ve, d_st, d_of, d_po);
  if (!rc) {
    cudaError_t e = cudaMemcpyAsync(out_status, d_st, Q, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out_offset, d_of, Q, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out_poses, d_po, Q * 64, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { ctx->err = std::string("mesh filter_host: ") + cudaGetErrorString(e); rc = CG_ECUDA; }
  }
  cg_voxels_destroy(vo);
  cg_voxels_destroy(ve);
  return rc;
}
