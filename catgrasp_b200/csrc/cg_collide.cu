// cg_collide.cu -- fused grasp-pose filter: pose composition + approach test +
// lateral-offset search + gripper-SDF collision predicate, one CTA per
// (grasp pose, symmetry) pair.
//
// Pose logic restates my_cpp/common.cpp:159,185-212,253-299 in the reference's
// fp32 operation order (Eigen 4x4 products without FMA contraction, column
// normalisation by division through sqrt, the float step accumulator whose 3 mm
// iteration never executes).  The geometry predicate replaces FCL
// mesh-vs-octree (collision_manager.cpp:93-111) with the SDF lookups of
// meshpy/meshpy/sdf.py:292-343 (trilinear) / :377-389 (nearest, in-bounds only):
// scene points are carried into the posed gripper's SDF grid and the pose
// collides iff any point has sd < 0.
//
// Every floating-point operation below is spelled with an explicit rounding
// intrinsic so that the CPU oracle (oracle/filter_ref.c) can reproduce the
// result bit for bit.
#include "cg_common.cuh"
#include "cg_pose.cuh"

struct cg_sdf {
  cg_ctx *ctx;
  float *grid;  // device, data[i][j][k]
  int nx, ny, nz;
  float origin[3];
  float res;
  int border_nonneg;   // every cell on the six boundary faces is >= 0 (true for padded grids, make_sdf.py:30)
  float border_min;    // smallest value on the six boundary faces
};

namespace {

struct SdfView {
  const float *grid;
  int nx, ny, nz;
  float ox, oy, oz;
  float inv_res;
  int border_nonneg;
};

using namespace cg_pose;

__device__ __forceinline__ float sdf_trilinear(const SdfView &s, float gx, float gy, float gz) {
  // sdf.py:311-343: clip, floor, 8 corners, out-of-bounds corners contribute 0
  const float cx = fminf(fmaxf(gx, 0.f), (float)(s.nx - 1));
  const float cy = fminf(fmaxf(gy, 0.f), (float)(s.ny - 1));
  const float cz = fminf(fmaxf(gz, 0.f), (float)(s.nz - 1));
  const float lx = floorf(cx), ly = floorf(cy), lz = floorf(cz);
  const int ix = (int)lx, iy = (int)ly, iz = (int)lz;
  // weight per axis: 1 - |corner - coord|
  const float wx0 = sub(1.f, sub(cx, lx)), wx1 = sub(1.f, sub(add(lx, 1.f), cx));
  const float wy0 = sub(1.f, sub(cy, ly)), wy1 = sub(1.f, sub(add(ly, 1.f), cy));
  const float wz0 = sub(1.f, sub(cz, lz)), wz1 = sub(1.f, sub(add(lz, 1.f), cz));
  const bool hx = (ix + 1) < s.nx, hy = (iy + 1) < s.ny, hz = (iz + 1) < s.nz;
  const size_t sx = (size_t)s.ny * s.nz, sy = (size_t)s.nz;
  const float *p = s.grid + (size_t)ix * sx + (size_t)iy * sy + iz;
  // corner order of Sdf3D (sdf.py:217-225): i -> (x,y,z) in {min,max}
  //   0:(0,0,0) 1:(1,0,0) 2:(0,1,0) 3:(0,0,1) 4:(1,1,0) 5:(0,1,1) 6:(1,0,1) 7:(1,1,1)
  const float v0 = __ldg(p);
  const float v1 = hx ? __ldg(p + sx) : 0.f;
  const float v2 = hy ? __ldg(p + sy) : 0.f;
  const float v3 = hz ? __ldg(p + 1) : 0.f;
  const float v4 = (hx && hy) ? __ldg(p + sx + sy) : 0.f;
  const float v5 = (hy && hz) ? __ldg(p + sy + 1) : 0.f;
  const float v6 = (hx && hz) ? __ldg(p + sx + 1) : 0.f;
  const float v7 = (hx && hy && hz) ? __ldg(p + sx + sy + 1) : 0.f;
  float sd = 0.f;
  sd = fmaf(mul(mul(wx0, wy0), wz0), v0, sd);
  sd = fmaf(mul(mul(wx1, wy0), wz0), v1, sd);
  sd = fmaf(mul(mul(wx0, wy1), wz0), v2, sd);
  sd = fmaf(mul(mul(wx0, wy0), wz1), v3, sd);
  sd = fmaf(mul(mul(wx1, wy1), wz0), v4, sd);
  sd = fmaf(mul(mul(wx0, wy1), wz1), v5, sd);
  sd = fmaf(mul(mul(wx1, wy0), wz1), v6, sd);
  sd = fmaf(mul(mul(wx1, wy1), wz1), v7, sd);
  return sd;
}

// nearest cell; *inb = false when the rounded cell is outside the grid
__device__ __forceinline__ float sdf_nearest(const SdfView &s, float gx, float gy, float gz, bool clamp, bool *inb) {
  float rx = rintf(gx), ry = rintf(gy), rz = rintf(gz);  // np.round / torch.round: half to even
  bool ok = (rx >= 0.f) && (rx < (float)s.nx) && (ry >= 0.f) && (ry < (float)s.ny) && (rz >= 0.f) && (rz < (float)s.nz);
  if (!ok) {
    if (!clamp) { *inb = false; return 0.f; }
    rx = fminf(fmaxf(rx, 0.f), (float)(s.nx - 1));
    ry = fminf(fmaxf(ry, 0.f), (float)(s.ny - 1));
    rz = fminf(fmaxf(rz, 0.f), (float)(s.nz - 1));
  }
  *inb = true;
  return __ldg(s.grid + ((size_t)(int)rx * s.ny + (int)ry) * s.nz + (int)rz);
}

// camera frame -> grid coordinates of one SDF in a single affine map: G = inv_res * (inv - origin)
// (sdf.py:252-264 folded into the inverse pose; rounding order fixed here and in oracle/filter_ref.c)
__device__ void fold_grid(const float *inv, const SdfView &s, float *out) {
#pragma unroll
  for (int k = 0; k < 9; k++) out[k] = mul(inv[k], s.inv_res);
  out[9] = mul(sub(inv[9], s.ox), s.inv_res);
  out[10] = mul(sub(inv[10], s.oy), s.inv_res);
  out[11] = mul(sub(inv[11], s.oz), s.inv_res);
}

// true iff point x (camera frame) lies inside the posed gripper: sd(G * x) < 0
__device__ __forceinline__ bool point_hits(const SdfView &s, const float *G, int mode, float margin, float x, float y, float z) {
  const float gx = fmaf(G[2], z, fmaf(G[1], y, fmaf(G[0], x, G[9])));
  const float gy = fmaf(G[5], z, fmaf(G[4], y, fmaf(G[3], x, G[10])));
  const float gz = fmaf(G[8], z, fmaf(G[7], y, fmaf(G[6], x, G[11])));
  if (mode == CG_SDF_TRILINEAR) {
    // Exact shortcut: a coordinate outside [0, dim-1] is clamped onto a boundary face (sdf.py:311-313) and then
    // interpolates boundary cells only; when all of those are >= 0 the result cannot be < 0, so the eight gathers
    // are skipped.  Most scene points are far from the gripper box, which makes this the common path.
    if (s.border_nonneg && (gx < 0.f || gy < 0.f || gz < 0.f || gx > (float)(s.nx - 1) || gy > (float)(s.ny - 1) ||
                            gz > (float)(s.nz - 1)))
      return false;
    return sdf_trilinear(s, gx, gy, gz) < margin;
  }
  bool inb;
  const float sd = sdf_nearest(s, gx, gy, gz, false, &inb);
  return inb && (sd < margin);
}

constexpr int FT = 256;

// Points whose trilinear lookup cannot be skipped are queued (grid coordinates) so that the eight-corner gather runs
// with full warps: most scene points miss the gripper's grid box, and evaluating the survivors in place left ~46 % of
// the lanes idle (ncu: 17.4 active threads per instruction).
constexpr int QCAP = 4 * FT;
struct HitQueue {
  float x[QCAP], y[QCAP], z[QCAP];
  int count[2];
};

// Scans points pts[0], pts[stride], ..., pts[(P-1)*stride] (rows of 3 floats).
__device__ bool any_point_hits(const SdfView &s, const float *G, int mode, float margin, const float *__restrict__ pts, int P,
                               int stride, volatile int *flag, HitQueue &Q) {
  // four independent points per thread and iteration (12 loads in flight) -- the loop is latency-bound otherwise;
  // within one j the 256 threads read consecutive points (coalesced 12-byte rows)
  if (!(mode == CG_SDF_TRILINEAR && s.border_nonneg)) {
    bool hit = false;
    for (int base = 0; base < P; base += 4 * FT) {
      float x[4], y[4], z[4];
      bool ok[4];
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const int p = base + j * FT + threadIdx.x;
        ok[j] = p < P;
        const size_t o = 3 * (size_t)(ok[j] ? p : 0) * (size_t)stride;
        x[j] = __ldg(pts + o); y[j] = __ldg(pts + o + 1); z[j] = __ldg(pts + o + 2);
      }
#pragma unroll
      for (int j = 0; j < 4; j++) hit = hit || (ok[j] && point_hits(s, G, mode, margin, x[j], y[j], z[j]));
      if (hit) { *flag = 1; break; }
      if (*flag) break;   // another thread already found a collision
    }
    return __syncthreads_or(hit) != 0;
  }
  // Trilinear with a non-negative border: the exact out-of-box shortcut of point_hits() decides most points; the rest
  // go through the queue.  Same arithmetic per point as point_hits(), so the verdict is unchanged.
  const float g0 = G[0], g1 = G[1], g2 = G[2], g3 = G[3], g4 = G[4], g5 = G[5], g6 = G[6], g7 = G[7], g8 = G[8];
  const float t0 = G[9], t1 = G[10], t2 = G[11];
  const float hx = (float)(s.nx - 1), hy = (float)(s.ny - 1), hz = (float)(s.nz - 1);
  const int lane = threadIdx.x & 31;
  const unsigned lt = (1u << lane) - 1u;
  int cur = 0;
  if (threadIdx.x == 0) { Q.count[0] = 0; Q.count[1] = 0; }
  __syncthreads();
  for (int base = 0; base < P; base += 4 * FT) {
    float x[4], y[4], z[4];
    bool ok[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int p = base + j * FT + threadIdx.x;
      ok[j] = p < P;
      const size_t o = 3 * (size_t)(ok[j] ? p : 0) * (size_t)stride;
      x[j] = __ldg(pts + o); y[j] = __ldg(pts + o + 1); z[j] = __ldg(pts + o + 2);
    }
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const float gx = fmaf(g2, z[j], fmaf(g1, y[j], fmaf(g0, x[j], t0)));
      const float gy = fmaf(g5, z[j], fmaf(g4, y[j], fmaf(g3, x[j], t1)));
      const float gz = fmaf(g8, z[j], fmaf(g7, y[j], fmaf(g6, x[j], t2)));
      const bool need = ok[j] && !(gx < 0.f || gy < 0.f || gz < 0.f || gx > hx || gy > hy || gz > hz);
      const unsigned m = __ballot_sync(0xffffffffu, need);
      if (m) {
        int at = 0;
        if (lane == 0) at = atomicAdd(&Q.count[cur], __popc(m));
        at = __shfl_sync(0xffffffffu, at, 0);
        if (need) {
          const int e = at + __popc(m & lt);
          Q.x[e] = gx; Q.y[e] = gy; Q.z[e] = gz;
        }
      }
    }
    __syncthreads();
    const int n = Q.count[cur];
    if (threadIdx.x == 0) Q.count[cur ^ 1] = 0;      // next chunk's counter; nobody touches it before the barrier below
    bool hit = false;
    for (int e = threadIdx.x; e < n; e += FT) hit = hit || (sdf_trilinear(s, Q.x[e], Q.y[e], Q.z[e]) < margin);
    if (__syncthreads_or(hit)) return true;
    cur ^= 1;
  }
  return false;
}

__global__ void __launch_bounds__(FT) filter_kernel(const cg_filter_params prm, const float *__restrict__ grasp_poses,
                                                    int G, const float *__restrict__ sym, int S, SdfView sdf_open,
                                                    const float *__restrict__ open_pts, int P1, SdfView sdf_encl,
                                                    const float *__restrict__ encl_pts, int P2,
                                                    uint8_t *__restrict__ out_status, int8_t *__restrict__ out_offset,
                                                    float *__restrict__ out_poses) {
  __shared__ float g_s[16];      // grasp_in_cam (normalised)
  __shared__ float cur_s[16];    // shifted candidate
  __shared__ float inv_s[12], go_s[12], ge_s[12];   // inverse gripper pose; folded camera->grid maps (open, enclosed)
  __shared__ int rej_dir;
  __shared__ int flag;
  __shared__ HitQueue hq;
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
  bool open_hit = false;
  int winner = -1;
  for (int k = 0; k < n_off; k++) {
    if (threadIdx.x == 0) {
      float cur[16], gic[16];
      offset_pose(g_s, k, prm.gripper_in_grasp, cur, gic);
      affine_inverse(gic, inv_s);
      fold_grid(inv_s, sdf_open, go_s);
      fold_grid(inv_s, sdf_encl, ge_s);
      for (int e = 0; e < 16; e++) cur_s[e] = cur[e];
      flag = 0;
    }
    __syncthreads();
    // The verdict is (open gripper hits the object's points) OR (swept gripper hits the background points), so the
    // order of the scans is free (the reference does open first, common.cpp:268-278).  In clutter nearly every rejection
    // comes from the background and shows up within a few hundred well-spread background points, whereas the object's own
    // points all lie inside the gripper's grid box (every one needs the eight-corner lookup) and never end the scan
    // early.  So: a strided sample of the background (every (P2/1024)-th point: spatially uniform whatever order the
    // caller's points come in -- raster order of an occupancy image, sorted, shuffled), then the object set, then the
    // whole background.  (`flag` is only ever set by a hit, so it is still clear whenever a later scan starts.)
    const int head = min(P2, 4 * FT);
    const int hstride = head > 0 ? P2 / head : 1;
    bool coll;
    if (split) {
      // the caller wants to know WHICH test rejected (verbose counters): the reference's order, open gripper first
      coll = any_point_hits(sdf_open, go_s, prm.sdf_mode, prm.sdf_margin, open_pts, P1, 1, &flag, hq);
      open_hit = coll;
      if (!coll && head > 0) coll = any_point_hits(sdf_encl, ge_s, prm.sdf_mode, prm.sdf_margin, encl_pts, head, hstride, &flag, hq);
    } else {
      coll = (head > 0) && any_point_hits(sdf_encl, ge_s, prm.sdf_mode, prm.sdf_margin, encl_pts, head, hstride, &flag, hq);
      if (!coll) coll = any_point_hits(sdf_open, go_s, prm.sdf_mode, prm.sdf_margin, open_pts, P1, 1, &flag, hq);
    }
    if (!coll && P2 > head) coll = any_point_hits(sdf_encl, ge_s, prm.sdf_mode, prm.sdf_margin, encl_pts, P2, 1, &flag, hq);
    if (!coll) { winner = k; break; }
    __syncthreads();  // everyone is done reading inv_s / flag before thread 0 rewrites them
  }
  if (threadIdx.x == 0) {
    out_status[q] = (winner >= 0) ? CG_ST_ACCEPT : ((split && !open_hit) ? CG_ST_REJ_COLL_ENCL : CG_ST_REJ_COLL);
    out_offset[q] = (int8_t)winner;
  }
  if (threadIdx.x < 16) out_poses[q * 16 + threadIdx.x] = (winner >= 0) ? cur_s[threadIdx.x] : 0.f;
}

__global__ void sdf_lookup_kernel(SdfView s, const float *__restrict__ gc, int P, int mode, float *__restrict__ out) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const float gx = gc[3 * (size_t)p], gy = gc[3 * (size_t)p + 1], gz = gc[3 * (size_t)p + 2];
  if (mode == CG_SDF_TRILINEAR) {
    out[p] = sdf_trilinear(s, gx, gy, gz);
  } else {
    bool inb;
    out[p] = sdf_nearest(s, gx, gy, gz, true, &inb);  // sdf.py:352-358 clamps
  }
}

SdfView make_view(const cg_sdf *s, float margin = 0.f) {
  SdfView v;
  v.grid = s->grid; v.nx = s->nx; v.ny = s->ny; v.nz = s->nz;
  v.ox = s->origin[0]; v.oy = s->origin[1]; v.oz = s->origin[2];
  v.inv_res = 1.0f / s->res;
  // the out-of-box shortcut stays exact as long as no boundary cell can report a hit: boundary values >= margin
  v.border_nonneg = (margin <= 0.f) ? s->border_nonneg : (s->border_min >= margin ? 1 : 0);
  return v;
}

}  // namespace

extern "C" int cg_sdf_create(cg_ctx *ctx, const float *grid_host, int nx, int ny, int nz, const float origin[3],
                             float resolution, cg_sdf **out) {
  if (!ctx || !out) return CG_EINVAL;
  CG_REQUIRE(ctx, grid_host && nx > 0 && ny > 0 && nz > 0 && resolution > 0.f, "sdf: bad grid");
  CG_CUDA(ctx, cudaSetDevice(ctx->device));
  cg_sdf *s = new cg_sdf();
  s->ctx = ctx; s->nx = nx; s->ny = ny; s->nz = nz; s->res = resolution;
  for (int k = 0; k < 3; k++) s->origin[k] = origin[k];
  const size_t bytes = (size_t)nx * ny * nz * sizeof(float);
  s->border_nonneg = 1;
  s->border_min = 3.0e38f;
  for (int i = 0; i < nx; i++)
    for (int j = 0; j < ny; j++)
      for (int k = 0; k < nz; k++) {
        if (i > 0 && i < nx - 1 && j > 0 && j < ny - 1 && k > 0 && k < nz - 1) { k = nz - 2; continue; }   // jump to the far face
        const float v = grid_host[((size_t)i * ny + j) * nz + k];
        if (!(v >= 0.f)) s->border_nonneg = 0;
        if (!(v >= s->border_min)) s->border_min = v;   // NaN counts as "smallest"
      }
  CG_CUDA(ctx, cudaMalloc(&s->grid, bytes));
  CG_CUDA(ctx, cudaMemcpyAsync(s->grid, grid_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
  CG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  *out = s;
  return CG_OK;
}

extern "C" void cg_sdf_destroy(cg_sdf *sdf) {
  if (!sdf) return;
  cudaSetDevice(sdf->ctx->device);
  cudaFree(sdf->grid);
  delete sdf;
}

extern "C" int cg_sdf_lookup_dev(cg_sdf *sdf, const float *grid_coords, int P, int mode, float *out_sd) {
  if (!sdf) return CG_EINVAL;
  cg_ctx *ctx = sdf->ctx;
  CG_REQUIRE(ctx, grid_coords && out_sd && P > 0, "sdf_lookup: bad arguments");
  CG_REQUIRE(ctx, mode == CG_SDF_TRILINEAR || mode == CG_SDF_NEAREST, "sdf_lookup: mode");
  sdf_lookup_kernel<<<(P + 255) / 256, 256, 0, ctx->stream>>>(make_view(sdf), grid_coords, P, mode, out_sd);
  CG_LAUNCH_CHECK(ctx);
  return CG_OK;
}

extern "C" int cg_filter_grasp_pose_dev(cg_ctx *ctx, const cg_filter_params *prm, const float *grasp_poses, int G,
                                        const float *symmetry_tfs, int S, cg_sdf *sdf_open, const float *open_pts,
                                        int P1, cg_sdf *sdf_enclosed, const float *enclosed_pts, int P2,
                                        uint8_t *out_status, int8_t *out_offset, float *out_poses) {
  if (!ctx) return CG_EINVAL;
  CG_REQUIRE(ctx, prm && grasp_poses && symmetry_tfs && G > 0 && S > 0, "filter: poses");
  CG_REQUIRE(ctx, sdf_open && (P1 == 0 || open_pts) && P1 >= 0, "filter: open gripper sdf/points");
  CG_REQUIRE(ctx, P2 == 0 || (sdf_enclosed && enclosed_pts), "filter: enclosed gripper sdf/points");
  CG_REQUIRE(ctx, out_status && out_offset && out_poses, "filter: outputs");
  CG_REQUIRE(ctx, prm->sdf_mode == CG_SDF_TRILINEAR || prm->sdf_mode == CG_SDF_NEAREST, "filter: sdf_mode");
  CG_REQUIRE(ctx, (long)G * S < 2147483647L, "filter: too many pairs");
  CG_REQUIRE(ctx, prm->sdf_margin >= 0.f && prm->sdf_margin < 1.f, "filter: sdf_margin (metres) out of range");
  CG_CUDA(ctx, cudaSetDevice(ctx->device));
  SdfView vo = make_view(sdf_open, prm->sdf_margin);
  SdfView ve = sdf_enclosed ? make_view(sdf_enclosed, prm->sdf_margin) : vo;
  filter_kernel<<<(unsigned)((long)G * S), FT, 0, ctx->stream>>>(*prm, grasp_poses, G, symmetry_tfs, S, vo, open_pts,
                                                                 P1, ve, enclosed_pts, P2, out_status, out_offset,
                                                                 out_poses);
  CG_LAUNCH_CHECK(ctx);
  return CG_OK;
}

extern "C" int cg_filter_grasp_pose_host(cg_ctx *ctx, const cg_filter_params *prm, const float *grasp_poses, int G,
                                         const float *symmetry_tfs, int S, cg_sdf *sdf_open, const float *open_pts,
                                         int P1, cg_sdf *sdf_enclosed, const float *enclosed_pts, int P2,
                                         uint8_t *out_status, int8_t *out_offset, float *out_poses) {
  if (!ctx) return CG_EINVAL;
  CG_REQUIRE(ctx, prm && grasp_poses && symmetry_tfs && G > 0 && S > 0, "filter_host: poses");
  CG_REQUIRE(ctx, out_status && out_offset && out_poses, "filter_host: outputs");
  CG_CUDA(ctx, cudaSetDevice(ctx->device));
  const size_t Q = (size_t)G * S;
  const size_t need = cg_arena::pad((size_t)G * 64) + cg_arena::pad((size_t)S * 64) + cg_arena::pad((size_t)P1 * 12) +
                      cg_arena::pad((size_t)P2 * 12) + cg_arena::pad(Q) * 2 + cg_arena::pad(Q * 64) + 4096;
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
  rc = cg_filter_grasp_pose_dev(ctx, prm, d_g, G, d_s, S, sdf_open, d_p1, P1, sdf_enclosed, d_p2, P2, d_st, d_of, d_po);
  if (rc) return rc;
  CG_CUDA(ctx, cudaMemcpyAsync(out_status, d_st, Q, cudaMemcpyDeviceToHost, st));
  CG_CUDA(ctx, cudaMemcpyAsync(out_offset, d_of, Q, cudaMemcpyDeviceToHost, st));
  CG_CUDA(ctx, cudaMemcpyAsync(out_poses, d_po, Q * 64, cudaMemcpyDeviceToHost, st));
  CG_CUDA(ctx, cudaStreamSynchronize(st));
  return CG_OK;
}
